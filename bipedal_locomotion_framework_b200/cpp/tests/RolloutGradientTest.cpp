/**
 * @file RolloutGradientTest.cpp
 * ContactRolloutBatch::rolloutCostGradient (the reverse mode of the fused rollout's cost; no
 * reference counterpart) against central differences of ContactRolloutBatch::rollout's costs, and
 * its argument checks.  Needs a GPU.
 */
#ifdef BLF_HAVE_CATCH2
#include <catch2/catch.hpp>
#else
#include "catch_shim.h"
#endif

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>

#include <BipedalLocomotion/ContactModels/ContinuousContactModelBatch.h>
#include <BipedalLocomotion/GenericContainer/DeviceSoA.h>
#include <BipedalLocomotion/System/ContactRolloutBatch.h>

#include "blf_ccm.h"

using namespace BipedalLocomotion::ContactModels;
using namespace BipedalLocomotion::System;
using BipedalLocomotion::GenericContainer::DeviceSoA;

namespace
{
constexpr std::size_t kRollouts = 8;
constexpr int kFeet = 2;
constexpr int kHorizon = 20;
constexpr std::size_t kChains = kRollouts * kFeet;
constexpr std::size_t kSteps = kChains * kHorizon;
constexpr double kDT = 0.01, kRho = 0.05;

struct Rng
{
    std::uint64_t s = 0x2545F4914F6CDD1Dull;
    double uniform(double lo, double hi)
    {
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        return lo + (hi - lo) * double(s >> 11) * (1.0 / 9007199254740992.0);
    }
};

void rpy(double r, double p, double y, double* R)
{
    const double cr = std::cos(r), sr = std::sin(r), cp = std::cos(p), sp = std::sin(p);
    const double cy = std::cos(y), sy = std::sin(y);
    const double m[9] = {cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr,
                         sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr,
                         -sp,     cp * sr,                cp * cr};
    std::copy(m, m + 9, R);
}

struct Host
{
    std::vector<std::vector<double>> twists, positions, rotations, nulls;
};

Host makeInputs()
{
    Rng rng;
    Host h{std::vector<std::vector<double>>(6, std::vector<double>(kSteps)),
           std::vector<std::vector<double>>(3, std::vector<double>(kChains)),
           std::vector<std::vector<double>>(9, std::vector<double>(kChains)),
           std::vector<std::vector<double>>(12, std::vector<double>(kChains))};
    for (std::size_t i = 0; i < kSteps; ++i)
        for (int j = 0; j < 6; ++j) h.twists[j][i] = rng.uniform(-0.2, 0.2);
    for (std::size_t c = 0; c < kChains; ++c)
    {
        double R[9], R0[9];
        rpy(rng.uniform(-0.3, 0.3) + (c % 5 == 1 ? 3.0 : 0.0), rng.uniform(-0.3, 0.3), rng.uniform(-3.0, 3.0), R);
        rpy(rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05), rng.uniform(-3.0, 3.0), R0);
        for (int j = 0; j < 3; ++j)
        {
            h.positions[j][c] = rng.uniform(-0.01, 0.01);
            h.nulls[j][c] = h.positions[j][c] + rng.uniform(-0.005, 0.005);
        }
        for (int j = 0; j < 9; ++j)
        {
            h.rotations[j][c] = R[j];
            h.nulls[3 + j][c] = R0[j];
        }
    }
    return h;
}

bool upload(DeviceSoA& d, const std::vector<std::vector<double>>& h)
{
    for (std::size_t p = 0; p < h.size(); ++p)
        if (!d.upload(p, h[p].data())) return false;
    return true;
}

std::vector<std::vector<double>> download(const DeviceSoA& d)
{
    std::vector<std::vector<double>> h(d.planes(), std::vector<double>(d.size()));
    for (std::size_t p = 0; p < d.planes(); ++p) d.download(p, h[p].data());
    return h;
}
} // namespace

TEST_CASE("rolloutCostGradient agrees with central differences of rollout")
{
    auto device = CudaDevice::open(0);
    REQUIRE(device != nullptr);
    REQUIRE(blf_ccm_set_uniform_params(static_cast<blf_ccm_handle*>(device->handle()), 0.2, 0.1, 2000.0, 50.0) == 0);
    ContactRolloutBatch rollouts(device);
    Host h = makeInputs();
    DeviceSoA twists(device, 6, kSteps), positions(device, 3, kChains), rotations(device, 9, kChains);
    DeviceSoA nulls(device, 12, kChains), costPlane(device, 1, kRollouts), bestPlane(device, 1, 2);
    DeviceSoA gradCost(device, 1, kRollouts);
    DeviceSoA gTwist(device, 6, kSteps), gPos(device, 3, kChains), gRot(device, 9, kChains);
    DeviceSoA gNull(device, 12, kChains), gParams(device, 4, kChains);
    REQUIRE(upload(twists, h.twists));
    REQUIRE(upload(positions, h.positions));
    REQUIRE(upload(rotations, h.rotations));
    REQUIRE(upload(nulls, h.nulls));
    std::vector<double> gbar(kRollouts);
    Rng rng;
    for (auto& g : gbar) g = rng.uniform(0.5, 2.0);
    REQUIRE(gradCost.upload(0, gbar.data()));
    iDynTree::Wrench reference;
    reference(2) = 5.0;
    REQUIRE(rollouts.rolloutCostGradient(kRollouts, kFeet, kHorizon, kDT, kRho, twists, positions, rotations,
                                         nulls, nullptr, reference, 1.0, 10.0, gradCost.plane(0), &gTwist, &gPos,
                                         &gRot, &gNull, &gParams));
    const auto gt = download(gTwist), gp = download(gPos), gr = download(gRot);

    auto weighted = [&]() {
        std::vector<double> c(kRollouts);
        rollouts.rollout(kRollouts, kFeet, kHorizon, kDT, kRho, twists, positions, rotations, nulls, nullptr,
                         0u, nullptr, nullptr, nullptr, nullptr, nullptr, reference, 1.0, 10.0, 0,
                         costPlane.plane(0), bestPlane.plane(0));
        costPlane.download(0, c.data());
        double s = 0.0;
        for (std::size_t r = 0; r < kRollouts; ++r) s += gbar[r] * c[r];
        return s;
    };
    // one coordinate of a plane, perturbed by +-h: (s(x+h) - s(x-h)) / 2h
    auto fd = [&](DeviceSoA& d, std::vector<std::vector<double>>& host, int plane, std::size_t i) {
        const double x = host[plane][i], step = 1e-6 * std::max(1.0, std::fabs(x));
        host[plane][i] = x + step;
        d.upload(plane, host[plane].data());
        const double up = weighted();
        host[plane][i] = x - step;
        d.upload(plane, host[plane].data());
        const double down = weighted();
        host[plane][i] = x;
        d.upload(plane, host[plane].data());
        return (up - down) / (2.0 * step);
    };
    double worst = 0.0, scale = 0.0;
    for (const auto* g : {&gt, &gp, &gr})
        for (const auto& plane : *g)
            for (double v : plane) scale = std::max(scale, std::fabs(v));
    for (std::size_t c = 0; c < kChains; c += 3)
        for (int t : {0, kHorizon / 2, kHorizon - 1})
            for (int j = 0; j < 6; ++j)
            {
                const std::size_t i = static_cast<std::size_t>(t) * kChains + c;
                worst = std::max(worst, std::fabs(fd(twists, h.twists, j, i) - gt[j][i]));
            }
    for (std::size_t c = 0; c < kChains; c += 5)
    {
        for (int j = 0; j < 3; ++j) worst = std::max(worst, std::fabs(fd(positions, h.positions, j, c) - gp[j][c]));
        for (int j = 0; j < 9; ++j) worst = std::max(worst, std::fabs(fd(rotations, h.rotations, j, c) - gr[j][c]));
    }
    REQUIRE(scale > 0.0);
    REQUIRE(worst <= 1e-5 * scale);
    const auto gn = download(gNull);
    for (int dead : {5, 8, 11})
        for (std::size_t c = 0; c < kChains; ++c) REQUIRE(gn[dead][c] == 0.0 && !std::signbit(gn[dead][c]));
}

TEST_CASE("rolloutCostGradient rejects mismatched containers")
{
    auto device = CudaDevice::open(0);
    REQUIRE(device != nullptr);
    REQUIRE(blf_ccm_set_uniform_params(static_cast<blf_ccm_handle*>(device->handle()), 0.2, 0.1, 2000.0, 50.0) == 0);
    ContactRolloutBatch rollouts(device);
    DeviceSoA twists(device, 6, kSteps), positions(device, 3, kChains), rotations(device, 9, kChains);
    DeviceSoA nulls(device, 12, kChains), gradCost(device, 1, kRollouts);
    DeviceSoA gTwist(device, 6, kSteps), shortTwist(device, 6, kSteps - 1), gPos(device, 3, kChains);
    iDynTree::Wrench reference;
    auto call = [&](DeviceSoA* gt, DeviceSoA* gp, DeviceSoA* gr) {
        return rollouts.rolloutCostGradient(kRollouts, kFeet, kHorizon, kDT, kRho, twists, positions, rotations,
                                            nulls, nullptr, reference, 1.0, 1.0, gradCost.plane(0), gt, gp, gr,
                                            nullptr, nullptr);
    };
    REQUIRE(call(&gTwist, nullptr, nullptr));
    REQUIRE_FALSE(call(&shortTwist, nullptr, nullptr));
    REQUIRE_FALSE(call(nullptr, nullptr, nullptr));   // nothing requested
    REQUIRE_FALSE(call(nullptr, &gPos, nullptr));     // positions without rotations
}
