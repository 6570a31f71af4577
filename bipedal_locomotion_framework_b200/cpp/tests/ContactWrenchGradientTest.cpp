/**
 * @file ContactWrenchGradientTest.cpp
 * ContinuousContactModelBatch::wrenchGradient (the reverse mode of the contact wrench; no reference
 * counterpart) against central differences of ContinuousContactModelBatch::evaluate, against the
 * regressor for the spring and damper gradients, and its argument checks.  Needs a GPU.
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

#include "blf_ccm.h"

using namespace BipedalLocomotion::ContactModels;
using BipedalLocomotion::GenericContainer::DeviceSoA;

namespace
{
constexpr std::size_t kN = 96;

struct Rng
{
    std::uint64_t s = 0x9E3779B97F4A7C15ull;
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

// host planes [30][kN]: near-flat feet, a few inverted ones
std::vector<std::vector<double>> makeStates()
{
    Rng rng;
    std::vector<std::vector<double>> x(30, std::vector<double>(kN));
    for (std::size_t i = 0; i < kN; ++i)
    {
        double R[9], R0[9];
        const double yaw = rng.uniform(-3.0, 3.0);
        rpy(rng.uniform(-0.3, 0.3) + (i % 7 == 0 ? 3.0 : 0.0), rng.uniform(-0.3, 0.3), yaw, R);
        rpy(rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05), yaw + rng.uniform(-0.1, 0.1), R0);
        for (int j = 0; j < 6; ++j) x[j][i] = rng.uniform(-1.0, 1.0);
        for (int j = 0; j < 3; ++j)
        {
            x[6 + j][i] = rng.uniform(-0.05, 0.05);
            x[18 + j][i] = x[6 + j][i] + rng.uniform(-0.01, 0.01);
        }
        for (int j = 0; j < 9; ++j)
        {
            x[9 + j][i] = R[j];
            x[21 + j][i] = R0[j];
        }
    }
    return x;
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

TEST_CASE("wrenchGradient agrees with central differences of evaluate")
{
    auto device = CudaDevice::open(0);
    REQUIRE(device != nullptr);
    ContinuousContactModelBatch batch(device);
    const auto host = makeStates();
    Rng rng;
    std::vector<std::vector<double>> cot(6, std::vector<double>(kN));
    std::vector<std::vector<double>> prm(4, std::vector<double>(kN));
    for (std::size_t i = 0; i < kN; ++i)
    {
        for (int r = 0; r < 6; ++r) cot[r][i] = rng.uniform(-1.0, 1.0);
        prm[0][i] = rng.uniform(0.08, 0.3);
        prm[1][i] = rng.uniform(0.04, 0.15);
        prm[2][i] = rng.uniform(1e3, 1e4);
        prm[3][i] = rng.uniform(10.0, 300.0);
    }
    DeviceSoA states(device, 30, kN), params(device, 4, kN), cotangent(device, 6, kN);
    DeviceSoA grad(device, 30, kN), gradParams(device, 4, kN), wrench(device, 6, kN);
    REQUIRE(upload(states, host));
    REQUIRE(upload(params, prm));
    REQUIRE(upload(cotangent, cot));
    REQUIRE(batch.wrenchGradient(states, &params, cotangent, &grad, &gradParams));
    const auto g = download(grad);
    const auto gp = download(gradParams);

    // gbar . (W(x + h e_j) - W(x - h e_j)) / 2h for every input plane and parameter
    auto projected = [&](std::vector<std::vector<double>>& x, std::vector<std::vector<double>>& q,
                         std::vector<double>& plane, std::vector<double>& out) {
        const std::vector<double> base = plane;
        std::vector<double> step(kN);
        std::vector<std::vector<double>> w[2];
        for (int side = 0; side < 2; ++side)
        {
            for (std::size_t i = 0; i < kN; ++i)
            {
                step[i] = 1e-6 * std::max(1.0, std::fabs(base[i]));
                plane[i] = base[i] + (side == 0 ? step[i] : -step[i]);
            }
            upload(states, x);
            upload(params, q);
            batch.evaluate(states, &params, ContinuousContactModelBatch::ContactWrench, &wrench, nullptr,
                           nullptr, nullptr);
            w[side] = download(wrench);
        }
        plane = base;
        for (std::size_t i = 0; i < kN; ++i)
        {
            out[i] = 0.0;
            for (int r = 0; r < 6; ++r) out[i] += cot[r][i] * (w[0][r][i] - w[1][r][i]) / (2.0 * step[i]);
        }
    };
    auto x = host;
    auto q = prm;
    std::vector<double> fd(kN);
    double worst = 0.0;
    auto compare = [&](const std::vector<double>& analytic) {
        for (std::size_t i = 0; i < kN; ++i)
        {
            if (std::fabs(host[17][i]) < 1e-4) continue; // the |R22| kink
            worst = std::max(worst, std::fabs(analytic[i] - fd[i]) / std::max(1.0, std::fabs(analytic[i])));
        }
    };
    for (int p = 0; p < 30; ++p)
    {
        projected(x, q, x[p], fd);
        compare(g[p]);
    }
    for (int p = 0; p < 4; ++p)
    {
        projected(x, q, q[p], fd);
        compare(gp[p]);
    }
    REQUIRE(worst < 1e-5);
    for (int dead : {11, 14, 23, 26, 29})
        for (std::size_t i = 0; i < kN; ++i) REQUIRE(g[dead][i] == 0.0 && !std::signbit(g[dead][i]));
}

TEST_CASE("wrenchGradient: spring and damper gradients are the regressor columns")
{
    auto device = CudaDevice::open(0);
    REQUIRE(device != nullptr);
    ContinuousContactModelBatch batch(device);
    REQUIRE(blf_ccm_set_uniform_params(static_cast<blf_ccm_handle*>(device->handle()), 0.12, 0.09, 2000.0, 100.0) == 0);
    DeviceSoA states(device, 30, kN), cotangent(device, 6, kN), gradParams(device, 4, kN), reg(device, 12, kN);
    REQUIRE(upload(states, makeStates()));
    REQUIRE(batch.evaluate(states, nullptr, ContinuousContactModelBatch::Regressor, nullptr, nullptr, nullptr, &reg));
    const auto y = download(reg);
    for (int r = 0; r < 6; ++r)
    {
        std::vector<std::vector<double>> cot(6, std::vector<double>(kN, 0.0));
        cot[r].assign(kN, 1.0);
        REQUIRE(upload(cotangent, cot));
        REQUIRE(batch.wrenchGradient(states, nullptr, cotangent, nullptr, &gradParams));
        const auto gp = download(gradParams);
        for (std::size_t i = 0; i < kN; ++i)
            for (int c = 0; c < 2; ++c)
            {
                // scale: the regressor's 3x1 block (force or torque rows) this entry belongs to
                double scale = 1e-300;
                for (int k = 3 * (r / 3); k < 3 * (r / 3) + 3; ++k) scale = std::max(scale, std::fabs(y[2 * k + c][i]));
                REQUIRE(std::fabs(gp[2 + c][i] - y[2 * r + c][i]) <= 1e-12 * scale);
            }
    }
}

TEST_CASE("wrenchGradient rejects mismatched containers")
{
    auto device = CudaDevice::open(0);
    REQUIRE(device != nullptr);
    ContinuousContactModelBatch batch(device);
    DeviceSoA states(device, 30, kN), cotangent(device, 6, kN), shortCotangent(device, 6, kN - 1);
    DeviceSoA grad(device, 30, kN), badGrad(device, 29, kN);
    REQUIRE_FALSE(batch.wrenchGradient(states, nullptr, shortCotangent, &grad, nullptr));
    REQUIRE_FALSE(batch.wrenchGradient(states, nullptr, cotangent, &badGrad, nullptr));
    REQUIRE_FALSE(batch.wrenchGradient(states, nullptr, cotangent, nullptr, nullptr)); // nothing requested
}
