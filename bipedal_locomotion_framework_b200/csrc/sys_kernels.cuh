// sys_kernels.cuh -- the steps either side of the contact model (SURVEY.md section 8(f) rows 2, 3).
//
//   kin_euler_step            FloatingBaseSystemKinematics::dynamics (base part) + one ForwardEuler
//                             step   src/System/src/FloatingBaseSystemKinematics.cpp:36-73,
//                             src/System/include/BipedalLocomotion/System/ForwardEuler.h:45-53
//   sys_kin_euler_kernel      that step for n independent systems, SoA planes (HBM-bound, 240 B)
//   sys_kin_aos_kernel        derivative / multi-step integrate for the per-instance facade
//   ccm_rollout_kernel        fused sampling-MPC rollout: one lane owns one (rollout, foot) chain,
//                             pose and null pose stay in registers for the whole horizon; per step
//                             only the 48-byte twist comes from HBM (cp.async ring, 8 steps ahead)
//                             -> contact model -> cost -> Euler step.  The 216 input bytes per
//                             evaluation of the unfused path never touch HBM; cost-only rollouts
//                             are FP64-pipe bound instead of HBM bound.
//   ccm_genforce_kernel       out[s] = base[s] + sum_c J_c^T wrench_c
//                             (src/System/src/FloatingBaseSystemDynamics.cpp:199-226): wrench in
//                             registers (never written to HBM unless asked), Jacobians streamed by
//                             TMA bulk copies through a per-warp ring, lanes own columns.
//
// Derivation differs from the oracle on purpose: Rdot's columns are w x c_j (not -(c_j x w) through
// a matrix), and the Baumgarte term uses (R R^T)^-1 R = R^-T = cofactors of R over det R instead of
// forming R R^T and inverting it with Eigen's general 3x3 formula.
#pragma once

#include <cuda.h>   // CUtensorMap (type only; the encoder is looked up at run time)

#include "ccm_kernels.cuh"

namespace blfccm {

// ------------------------------------------------------------------------------------------------
// kinematics
// ------------------------------------------------------------------------------------------------

struct Pose {
    V3 p;           // position
    V3 c0, c1, c2;  // columns of R
};

// 1/x to the last bit or two: the hardware's reciprocal seed (MUFU.RCP64H, ~20 bits) and two Newton
// steps.  An IEEE division costs 123 dependent cycles on B200 (tools/micro/fp64_lat.cu: DFMA 8.2,
// division 131 with its DADD, this sequence 47), and it sits on the sequential chain of every
// rollout step.  x = 0 gives NaN (inf from the seed, then 0 * inf), so a singular rotation still
// poisons the result as in the reference.
__device__ __forceinline__ double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}

// Rates of FloatingBaseSystemKinematics::dynamics (FloatingBaseSystemKinematics.cpp:59-66):
//   Rdot = -R.colwise().cross(w) + rho/2 ((R R^T)^-1 - I) R
// column by column: Rdot.col(j) = w x c_j + rho/2 (k_j / det R - c_j), because (R R^T)^-1 R = R^-T and
// the columns of R^-T are the cross products k_0 = c1 x c2, k_1 = c2 x c0, k_2 = c0 x c1 over
// det R = c0 . k_0 -- three cross products, one determinant and one reciprocal instead of forming
// R R^T, its adjugate and a 3x3 product.  Singular R gives NaN, as the reference.
template <bool BAUM>
__device__ __forceinline__ void kin_rates(const Pose& s, const V3& w, double half_rho, V3& d0,
                                          V3& d1, V3& d2)
{
    d0 = cross(w, s.c0);
    d1 = cross(w, s.c1);
    d2 = cross(w, s.c2);
    if constexpr (BAUM) {
        const V3 k0 = cross(s.c1, s.c2), k1 = cross(s.c2, s.c0), k2 = cross(s.c0, s.c1);
        const double det = s.c0.x * k0.x + s.c0.y * k0.y + s.c0.z * k0.z;
        const double g = half_rho * fast_rcp(det);          // rho/2 / det R
        d0 = d0 + (g * k0 - half_rho * s.c0);
        d1 = d1 + (g * k1 - half_rho * s.c1);
        d2 = d2 + (g * k2 - half_rho * s.c2);
    }
}

// One ForwardEuler step x += dx * dT (ForwardEuler.h:50) of that system.  The Baumgarte step is
// regrouped so that few operations depend on the reciprocal (it is the long pole of the chain):
//   c_j' = c_j + dT (w x c_j + g k_j - rho/2 c_j) = (1 - dT rho/2) c_j + dT (w x c_j) + (dT g) k_j
// i.e. everything but the last FMA per component is independent of 1/det.  75 FP64 instructions
// per step instead of ~95, critical path k -> det -> 1/det -> dT g -> FMA (about 13 dependent
// operations).  Every kernel integrates through this one function, so fused rollouts, the batched
// Euler step and the per-instance integrate agree bit for bit with one another; against the oracle
// (which follows Eigen's expression) the difference is a few ulp per step.
// One component of a rotation column's update, with the contraction spelled out so that every
// kernel rounds it the same way:  c' = beta k + (dT x + alpha c)   [ c' = dT x + c  without Baumgarte ]
template <bool BAUM>
__device__ __forceinline__ double kin_col_step(double c, double x, double k, double alpha, double beta, double dT)
{
    if constexpr (BAUM) return fma(beta, k, fma(dT, x, __dmul_rn(alpha, c)));
    else return fma(dT, x, c);
}

template <bool BAUM>
__device__ __forceinline__ V3 kin_col_step(const V3& c, const V3& x, const V3& k, double alpha, double beta, double dT)
{
    return V3{kin_col_step<BAUM>(c.x, x.x, k.x, alpha, beta, dT), kin_col_step<BAUM>(c.y, x.y, k.y, alpha, beta, dT),
              kin_col_step<BAUM>(c.z, x.z, k.z, alpha, beta, dT)};
}

// the two uniform factors of the regrouped Baumgarte step, rounded the same way wherever they are formed
__device__ __forceinline__ double kin_dthr(double dT, double half_rho) { return __dmul_rn(dT, half_rho); }
__device__ __forceinline__ double kin_alpha(double dT, double half_rho) { return __dsub_rn(1.0, __dmul_rn(dT, half_rho)); }

__device__ __forceinline__ double dot3(const V3& a, const V3& b) { return fma(a.z, b.z, fma(a.y, b.y, __dmul_rn(a.x, b.x))); }

template <bool BAUM>
__device__ __forceinline__ void kin_euler_step(Pose& s, const V3& v, const V3& w, double half_rho,
                                               double dT)
{
    s.p = V3{fma(dT, v.x, s.p.x), fma(dT, v.y, s.p.y), fma(dT, v.z, s.p.z)};
    const V3 x0 = cross(w, s.c0), x1 = cross(w, s.c1), x2 = cross(w, s.c2);
    V3 k0{}, k1{}, k2{};
    double alpha = 1.0, beta = 0.0;
    if constexpr (BAUM) {
        k0 = cross(s.c1, s.c2);
        k1 = cross(s.c2, s.c0);
        k2 = cross(s.c0, s.c1);
        alpha = kin_alpha(dT, half_rho);                     // uniform: hoisted out of every loop
        beta = __dmul_rn(kin_dthr(dT, half_rho), fast_rcp(dot3(s.c0, k0)));   // dT rho/2 / det R
    }
    s.c0 = kin_col_step<BAUM>(s.c0, x0, k0, alpha, beta, dT);
    s.c1 = kin_col_step<BAUM>(s.c1, x1, k1, alpha, beta, dT);
    s.c2 = kin_col_step<BAUM>(s.c2, x2, k2, alpha, beta, dT);
}

// Reverse mode of kin_euler_step, fast_rcp(x) differentiated as 1/x.  With alpha = kin_alpha,
// r = 1/det, beta = dT rho/2 r, k0 = c1 x c2, k1 = c2 x c0, k2 = c0 x c1, det = c0.k0:
//   c_j' = alpha c_j + dT w x c_j + beta k_j,  p' = p + dT v.
// On entry g holds the adjoint of the pose AFTER the step; on return the adjoint of the pose s before
// it, and gv, gw the step's contribution to the twist's adjoint (only formed when TW):
//   gv = dT p'bar     gw = dT sum_j c_j x c_j'bar     c_jbar = alpha c_j'bar + dT c_j'bar x w
//   k_jbar = beta c_j'bar,  betabar = sum_j c_j'bar.k_j,  detbar = -betabar beta r,  c_jbar += detbar k_j
//   and the cross products' adjoints: k0 feeds c1 (c2 x k0bar) and c2 (k0bar x c1), and so on.
// Without the Baumgarte term only the first three lines remain, with alpha = 1.
template <bool BAUM, bool TW>
__device__ __forceinline__ void kin_euler_step_vjp(const Pose& s, const V3& w, double half_rho, double dT,
                                                   Pose& g, V3& gv, V3& gw)
{
    const V3 b0 = g.c0, b1 = g.c1, b2 = g.c2;   // adjoints of the columns after the step
    if constexpr (TW) {
        gv = dT * g.p;
        gw = dT * (cross(s.c0, b0) + cross(s.c1, b1) + cross(s.c2, b2));
    }
    double alpha = 1.0;
    if constexpr (BAUM) alpha = kin_alpha(dT, half_rho);
    g.c0 = alpha * b0 + dT * cross(b0, w);
    g.c1 = alpha * b1 + dT * cross(b1, w);
    g.c2 = alpha * b2 + dT * cross(b2, w);
    if constexpr (BAUM) {
        const V3 k0 = cross(s.c1, s.c2), k1 = cross(s.c2, s.c0), k2 = cross(s.c0, s.c1);
        const double r = fast_rcp(dot3(s.c0, k0));
        const double beta = __dmul_rn(kin_dthr(dT, half_rho), r);
        const double gdet = -(dot3(b0, k0) + dot3(b1, k1) + dot3(b2, k2)) * beta * r;
        const V3 q0 = beta * b0, q1 = beta * b1, q2 = beta * b2;   // adjoints of k0, k1, k2
        g.c0 = g.c0 + gdet * k0 + cross(q1, s.c2) + cross(s.c1, q2);
        g.c1 = g.c1 + gdet * k1 + cross(s.c2, q0) + cross(q2, s.c0);
        g.c2 = g.c2 + gdet * k2 + cross(q0, s.c1) + cross(s.c0, q1);
    }
}

struct KinArgs {
    const double* tw[6];
    double* pos[3];   // in/out
    double* rot[9];   // in/out, row-major index
    double half_rho, dT;
    long long n;
};

template <bool BAUM>
__global__ void __launch_bounds__(128, 5)
sys_kin_euler_kernel(const __grid_constant__ KinArgs a)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    ptx::grid_dep_launch_dependents();   // PDL: see ccm_soa_kernel
    ptx::grid_dep_wait();
    if (i >= a.n) return;
    double t[6], x[12];
#pragma unroll
    for (int j = 0; j < 6; ++j) t[j] = __ldcs(a.tw[j] + i);
#pragma unroll
    for (int j = 0; j < 3; ++j) x[j] = __ldcs(a.pos[j] + i);
#pragma unroll
    for (int j = 0; j < 9; ++j) x[3 + j] = __ldcs(a.rot[j] + i);
    Pose s{V3{x[0], x[1], x[2]}, V3{x[3], x[6], x[9]}, V3{x[4], x[7], x[10]}, V3{x[5], x[8], x[11]}};
    kin_euler_step<BAUM>(s, V3{t[0], t[1], t[2]}, V3{t[3], t[4], t[5]}, a.half_rho, a.dT);
    __stcs(a.pos[0] + i, s.p.x); __stcs(a.pos[1] + i, s.p.y); __stcs(a.pos[2] + i, s.p.z);
    __stcs(a.rot[0] + i, s.c0.x); __stcs(a.rot[1] + i, s.c1.x); __stcs(a.rot[2] + i, s.c2.x);
    __stcs(a.rot[3] + i, s.c0.y); __stcs(a.rot[4] + i, s.c1.y); __stcs(a.rot[5] + i, s.c2.y);
    __stcs(a.rot[6] + i, s.c0.z); __stcs(a.rot[7] + i, s.c1.z); __stcs(a.rot[8] + i, s.c2.z);
}

// Per-instance facade kernel (array-of-structures, n is tiny): mode 0 = derivative only
// (pos_dot n*3, rot_dot n*9), mode 1 = `steps` Euler steps with a constant twist, the first
// steps-1 of size step_dT and the last of size last_dT (FixedStepIntegrator::integrate's schedule).
struct KinAosArgs {
    const double* twists;   // n*6
    double* pos;            // n*3   (mode 0: pos_dot out; mode 1: in/out)
    double* rot;            // n*9   (mode 1: in/out)
    const double* rot_in;   // mode 0: rotation in
    double* rot_dot;        // mode 0: out
    double half_rho, step_dT, last_dT;
    long long n;
    int steps;
    int mode;
};

template <bool BAUM>
__global__ void __launch_bounds__(128)
sys_kin_aos_kernel(const __grid_constant__ KinAosArgs a)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const double* T = a.twists + 6 * i;
    const V3 v{T[0], T[1], T[2]}, w{T[3], T[4], T[5]};
    const double* R = (a.mode == 0 ? a.rot_in : a.rot) + 9 * i;
    Pose s{V3{0.0, 0.0, 0.0}, V3{R[0], R[3], R[6]}, V3{R[1], R[4], R[7]}, V3{R[2], R[5], R[8]}};
    if (a.mode == 0) {
        V3 d0, d1, d2;
        kin_rates<BAUM>(s, w, a.half_rho, d0, d1, d2);
        double* o = a.rot_dot + 9 * i;
        o[0] = d0.x; o[1] = d1.x; o[2] = d2.x;
        o[3] = d0.y; o[4] = d1.y; o[5] = d2.y;
        o[6] = d0.z; o[7] = d1.z; o[8] = d2.z;
        a.pos[3 * i] = v.x; a.pos[3 * i + 1] = v.y; a.pos[3 * i + 2] = v.z;
        return;
    }
    s.p = V3{a.pos[3 * i], a.pos[3 * i + 1], a.pos[3 * i + 2]};
    for (int k = 0; k < a.steps - 1; ++k) kin_euler_step<BAUM>(s, v, w, a.half_rho, a.step_dT);
    kin_euler_step<BAUM>(s, v, w, a.half_rho, a.last_dT);
    a.pos[3 * i] = s.p.x; a.pos[3 * i + 1] = s.p.y; a.pos[3 * i + 2] = s.p.z;
    double* o = a.rot + 9 * i;
    o[0] = s.c0.x; o[1] = s.c1.x; o[2] = s.c2.x;
    o[3] = s.c0.y; o[4] = s.c1.y; o[5] = s.c2.y;
    o[6] = s.c0.z; o[7] = s.c1.z; o[8] = s.c2.z;
}

// joint positions: x += v * dT per step (elementwise, layout-agnostic)
__global__ void __launch_bounds__(256)
sys_axpy_steps_kernel(double* __restrict__ x, const double* __restrict__ v, long long n, int steps,
                      double step_dT, double last_dT)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double xi = x[i];
    const double vi = v[i];
    for (int k = 0; k < steps - 1; ++k) xi = xi + vi * step_dT;
    xi = xi + vi * last_dT;
    x[i] = xi;
}

// ------------------------------------------------------------------------------------------------
// fused rollout
// ------------------------------------------------------------------------------------------------

constexpr int kRolloutDepth = 8;                               // twist prefetch distance (steps)
constexpr int kRolloutRingBytes = kRolloutDepth * 6 * 32 * 8;  // per warp

struct RolloutArgs {
    const double* tw[6];     // [horizon*chains], index t*chains + chain
    const double* pos0[3];   // [chains]
    const double* rot0[9];
    const double* nul[12];   // null-force pose per chain: pos 0-2, rot row-major 3-11
    const double* prm[4];    // per-chain parameters (HET)
    double* pos_out[3];      // final pose (all NULL when not wanted; may alias pos0/rot0)
    double* rot_out[9];
    double* wrench[6];       // [horizon*chains]
    double* autodyn[6];
    double* ctrl;            // [horizon*chains][36]
    double* chain_cost;      // [chains]
    Prm uni;
    double ref[6];
    double wf, wt;
    double half_rho, dT;
    long long chains;
    int horizon;
    int ctrl_bulk;
    int write_final;
    int split;               // warps sharing one 32-chain tile (power of two, 1 = none)
    int t_base;              // global index of this launch's first step (time-chunked rollouts)
    int accumulate;          // chain_cost holds the cost of the steps before t_base: add to it
    // ccm_rollout_ws3_kernel only: TMA descriptors of the six twist planes ([horizon][chains] doubles,
    // box = kWs3BoxSteps x 32) and the fused reduction / arg-min / peer exchange
    CUtensorMap twmap[6];
    double* cost;            // [n_rollouts] or nullptr
    CostIdx* block_best;     // gridDim.x entries (handle scratch)
    unsigned int* counter;   // zero before launch; reset by the last CTA
    CostIdx* best;
    long long n_rollouts, index_base;
    int feet;
    P2pArgs p2p;             // nranks > 0: the last CTA also runs the peer exchange -> p2p.out
};

// Few chains (a sampling-MPC batch of configs[2] size is 8 192 chains = 256 warps for 592 warp
// schedulers) leave the FP64 pipes idle and the step latency exposed.  `split` = K > 1 lets K warps
// share the same 32 chains: every warp integrates the poses of all steps (cheap: ~35 FP64
// instructions per step) but evaluates the contact model and the cost only for the steps
// t = phase (mod K), so the per-warp critical path shrinks ~2-3x while the idle schedulers fill up.
// Each (chain, phase) writes its own partial cost: chain_cost[chain*K + phase]; the reduce kernel
// sums a rollout's feet*K partials in index order (deterministic for a given shape and device).
template <unsigned OUT, bool HET, bool BAUM>
__global__ void __launch_bounds__(256)
ccm_rollout_kernel(const __grid_constant__ RolloutArgs a)
{
    constexpr unsigned MASK = OUT | M_WRENCH;   // the cost needs the wrench
    constexpr int D = kRolloutDepth;
    constexpr int kPerWarp = kRolloutRingBytes + ((OUT & M_CTRL) ? kWarp * 288 : 0);
    extern __shared__ __align__(128) unsigned char smem_raw[];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int K = a.split;                      // power of two
    const long long gw = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp;
    const int phase = static_cast<int>(gw & (K - 1));
    const long long wbase = (gw / K) * kWarp;
    if (wbase >= a.chains) return;  // warp-uniform
    const long long c = wbase + lane;
    const bool on = c < a.chains;
    const int cnt = static_cast<int>(min64(kWarp, a.chains - wbase));
    const int H = a.horizon;

    double* ring = reinterpret_cast<double*>(smem_raw + static_cast<size_t>(warp) * kPerWarp);
    double* ctile = ring + D * 6 * kWarp;
    const uint32_t ring_s = ptx::smem_addr(ring) + static_cast<uint32_t>(lane) * 8u;

    // every lane stages its own six twist components of step t; nobody else reads them
    auto issue = [&](int t) {
        if (on && t < H) {
            const uint32_t dst = ring_s + static_cast<uint32_t>((t & (D - 1)) * 6 * kWarp * 8);
            const long long src = static_cast<long long>(t) * a.chains + c;
#pragma unroll
            for (int j = 0; j < 6; ++j) ptx::cp_async8(dst + j * kWarp * 8, a.tw[j] + src);
        }
        ptx::cp_async_commit();
    };
    // No programmatic dependent launch here (measured: 43 -> 70 us at 8 192 chains): this kernel
    // is latency-bound with about one working warp per scheduler, and the early-resident CTAs of
    // the next launches, parked in griddepcontrol.wait, take issue slots from it.
#pragma unroll
    for (int t = 0; t < D; ++t) issue(t);

    // chain constants
    Pose s{};
    V3 p0{}, n1{}, n2{};
    Prm q = a.uni;
    if (on) {
        s.p = V3{__ldg(a.pos0[0] + c), __ldg(a.pos0[1] + c), __ldg(a.pos0[2] + c)};
        s.c0 = V3{__ldg(a.rot0[0] + c), __ldg(a.rot0[3] + c), __ldg(a.rot0[6] + c)};
        s.c1 = V3{__ldg(a.rot0[1] + c), __ldg(a.rot0[4] + c), __ldg(a.rot0[7] + c)};
        s.c2 = V3{__ldg(a.rot0[2] + c), __ldg(a.rot0[5] + c), __ldg(a.rot0[8] + c)};
        p0 = V3{__ldg(a.nul[0] + c), __ldg(a.nul[1] + c), __ldg(a.nul[2] + c)};
        n1 = V3{__ldg(a.nul[3] + c), __ldg(a.nul[6] + c), __ldg(a.nul[9] + c)};
        n2 = V3{__ldg(a.nul[4] + c), __ldg(a.nul[7] + c), __ldg(a.nul[10] + c)};
        if constexpr (HET)
            q = make_prm(__ldg(a.prm[0] + c), __ldg(a.prm[1] + c), __ldg(a.prm[2] + c),
                         __ldg(a.prm[3] + c));
    }
    if constexpr ((OUT & M_CTRL) != 0) {
        double2* z = reinterpret_cast<double2*>(ctile);
#pragma unroll
        for (int j = 0; j < 18; ++j) z[lane + j * kWarp] = make_double2(0.0, 0.0);
        __syncwarp();
    }

    double acc = (a.accumulate && on) ? a.chain_cost[c * K + phase] : 0.0;
    bool staged = false;   // a ctrl tile of this warp may still be leaving shared memory
    for (int t = 0; t < H; ++t) {
        ptx::cp_async_wait<D - 1>();
        V3 v{}, w{};
        if (on) {
            const double* r = ring + (t & (D - 1)) * 6 * kWarp + lane;
            v = V3{r[0], r[kWarp], r[2 * kWarp]};
            w = V3{r[3 * kWarp], r[4 * kWarp], r[5 * kWarp]};
        }
        if (((a.t_base + t) & (K - 1)) == phase) {   // warp-uniform: this warp's share of the evaluations
        State st;
        st.v = v; st.w = w; st.p = s.p; st.p0 = p0;
        st.e1 = s.c0; st.e2 = s.c1;
        st.R02 = s.c2.x; st.R12 = s.c2.y; st.R22 = s.c2.z;
        st.n1 = n1; st.n2 = n2;
        Result r;
        eval_contact<MASK>(st, q, r);

        const long long i = static_cast<long long>(t) * a.chains + c;
        if constexpr ((OUT & M_CTRL) != 0) {
            // previous step's tile must have left shared memory before it is overwritten
            if (staged && a.ctrl_bulk && lane == 0) ptx::bulk_wait_read_all();
            __syncwarp();
            staged = true;
        }
        if (on) {
            if constexpr ((OUT & M_WRENCH) != 0) {
                __stcs(a.wrench[0] + i, r.force.x); __stcs(a.wrench[1] + i, r.force.y);
                __stcs(a.wrench[2] + i, r.force.z); __stcs(a.wrench[3] + i, r.torque.x);
                __stcs(a.wrench[4] + i, r.torque.y); __stcs(a.wrench[5] + i, r.torque.z);
            }
            if constexpr ((OUT & M_AUTODYN) != 0) {
                __stcs(a.autodyn[0] + i, r.fhead.x); __stcs(a.autodyn[1] + i, r.fhead.y);
                __stcs(a.autodyn[2] + i, r.fhead.z); __stcs(a.autodyn[3] + i, r.ftail.x);
                __stcs(a.autodyn[4] + i, r.ftail.y); __stcs(a.autodyn[5] + i, r.ftail.z);
            }
            if constexpr ((OUT & M_CTRL) != 0) stage_ctrl(ctile + lane * 36, r);
            const V3 df = r.force - V3{a.ref[0], a.ref[1], a.ref[2]};
            const V3 dt = r.torque - V3{a.ref[3], a.ref[4], a.ref[5]};
            acc = acc + (a.wf * (df.x * df.x + df.y * df.y + df.z * df.z) +
                         a.wt * (dt.x * dt.x + dt.y * dt.y + dt.z * dt.z));
        }
        if constexpr ((OUT & M_CTRL) != 0)
            flush_ctrl_tile(a.ctrl, ctile, static_cast<long long>(t) * a.chains + wbase, cnt, lane,
                            a.ctrl_bulk != 0);
        }

        kin_euler_step<BAUM>(s, v, w, a.half_rho, a.dT);
        issue(t + D);   // the slot just consumed
    }

    if (on) {
        a.chain_cost[c * K + phase] = acc;
        if (a.write_final && phase == 0) {
            a.pos_out[0][c] = s.p.x; a.pos_out[1][c] = s.p.y; a.pos_out[2][c] = s.p.z;
            a.rot_out[0][c] = s.c0.x; a.rot_out[1][c] = s.c1.x; a.rot_out[2][c] = s.c2.x;
            a.rot_out[3][c] = s.c0.y; a.rot_out[4][c] = s.c1.y; a.rot_out[5][c] = s.c2.y;
            a.rot_out[6][c] = s.c0.z; a.rot_out[7][c] = s.c1.z; a.rot_out[8][c] = s.c2.z;
        }
    }
    ptx::cp_async_wait<0>();
    if constexpr ((OUT & M_CTRL) != 0) {
        if (staged && a.ctrl_bulk && lane == 0) ptx::bulk_wait_read_all();
    }
}

// ------------------------------------------------------------------------------------------------
// Reverse mode of the fused rollout's cost (blf_ccm_rollout_cost_vjp): for cotangents gbar[r] of
// cost[r], gbar^T dcost/d(twists, initial pose, null pose, parameters).  One lane per chain, one
// 32-chain tile per warp, as ccm_rollout_kernel.
//   forward   the pose recurrence alone (no wrench), twists through a per-lane cp.async ring S steps
//             deep; the pose before every step t = kS (k < last segment) goes to the tape
//             ([k][12][chains], time-major, coalesced); the last segment's pose stays in registers
//             and its twists in the ring.
//   reverse   segment by segment from the last: the segment's poses are recomputed from its
//             checkpoint with kin_euler_step (bit-identical to the forward rollout) into shared
//             memory, then t = end .. start: wrench at (twist_t, pose_t), cotangent
//             (gF, gT) = 2 gbar (wf (F - Fref), wt (T - Tref)), the pose adjoint back through Euler
//             step t (kin_euler_step_vjp; step H-1 does not enter the cost), plus vjp_wrench at step
//             t; the twist gradient of step t is written.  Null-pose and parameter adjoints add up
//             in registers; after t = 0 the pose adjoint is the initial pose's gradient.
// The previous segment's twists are staged while this one is walked: slot sigma_k(j) holds step
// kS + j, with sigma alternating between j and S-1-j from segment to segment, so the slot a step
// frees during the backward walk is the one the previous segment's forward recompute needs next.
// Accumulations are rounded on their own (__dadd_rn): vjp_wrench's products are never contracted
// into them, so at H = 1 the result is blf_ccm_wrench_vjp_soa's, bit for bit.
// ------------------------------------------------------------------------------------------------

constexpr int kVjpSeg = 8;   // steps per tape segment (measured: profiles/r05_rollout_vjp_probe.log)

struct RolloutVjpArgs {
    const double* tw[6];      // [horizon*chains], index t*chains + chain
    const double* pos0[3];    // [chains]
    const double* rot0[9];
    const double* nul[12];
    const double* prm[4];     // per-chain parameters (HET)
    const double* gcost;      // [n_rollouts]
    double* gtw[6];           // [horizon*chains]   (G_TWIST)
    double* gpos[3];          // [chains]           (G_POSE)
    double* grot[9];
    double* gnul[12];         // [chains]           (G_NULL)
    double* gprm[4];          // [chains]           (G_PARAMS)
    double* tape;             // [segments-1][12][chains]
    double uni[4];            // uniform length, width, spring, damper
    double ref[6];
    double wf, wt;
    double half_rho, dT;
    long long chains;
    int horizon;
    int feet;
};

__device__ __forceinline__ V3 add_rn(const V3& a, const V3& b)
{
    return V3{__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y), __dadd_rn(a.z, b.z)};
}

template <bool HET, bool BAUM, unsigned GROUPS, int S>
__global__ void __launch_bounds__(32)
ccm_rollout_vjp_kernel(const __grid_constant__ RolloutVjpArgs a)
{
    static_assert(S >= 2 && (S & (S - 1)) == 0, "segment length: a power of two");
    constexpr bool kTw = (GROUPS & G_TWIST) != 0;
    constexpr bool kAdj = (GROUPS & (G_TWIST | G_POSE)) != 0;   // the pose adjoint recurrence is needed
    constexpr unsigned W = GROUPS | (kAdj ? G_POSE : 0u);         // groups of the per-step wrench VJP
    extern __shared__ __align__(128) unsigned char smem_raw[];

    const int lane = threadIdx.x & 31;
    const long long c = static_cast<long long>(blockIdx.x) * kWarp + lane;
    if (c >= a.chains) return;   // no warp-collective operation below: idle lanes leave
    const long long N = a.chains;
    const int H = a.horizon;

    double* ring = reinterpret_cast<double*>(smem_raw);   // [S][6][32] twists
    double* poses = ring + S * 6 * kWarp;                 // [S][12][32] the segment's poses
    const uint32_t ring_s = ptx::smem_addr(ring) + static_cast<uint32_t>(lane) * 8u;
    auto stage = [&](int t, int slot) {
        const uint32_t dst = ring_s + static_cast<uint32_t>(slot * 6 * kWarp * 8);
        const long long src = static_cast<long long>(t) * N + c;
#pragma unroll
        for (int j = 0; j < 6; ++j) ptx::cp_async8(dst + j * kWarp * 8, a.tw[j] + src);
    };
    auto twist = [&](int slot, V3& v, V3& w) {
        const double* r = ring + slot * 6 * kWarp + lane;
        v = V3{r[0], r[kWarp], r[2 * kWarp]};
        w = V3{r[3 * kWarp], r[4 * kWarp], r[5 * kWarp]};
    };
    // plain launch: as ccm_rollout_kernel (latency-bound, PDL measured worse there)
#pragma unroll
    for (int t = 0; t < S; ++t) {
        if (t < H) stage(t, t);
        ptx::cp_async_commit();
    }

    Pose s;
    s.p = V3{__ldg(a.pos0[0] + c), __ldg(a.pos0[1] + c), __ldg(a.pos0[2] + c)};
    s.c0 = V3{__ldg(a.rot0[0] + c), __ldg(a.rot0[3] + c), __ldg(a.rot0[6] + c)};
    s.c1 = V3{__ldg(a.rot0[1] + c), __ldg(a.rot0[4] + c), __ldg(a.rot0[7] + c)};
    s.c2 = V3{__ldg(a.rot0[2] + c), __ldg(a.rot0[5] + c), __ldg(a.rot0[8] + c)};
    const V3 p0{__ldg(a.nul[0] + c), __ldg(a.nul[1] + c), __ldg(a.nul[2] + c)};
    const V3 n1{__ldg(a.nul[3] + c), __ldg(a.nul[6] + c), __ldg(a.nul[9] + c)};
    const V3 n2{__ldg(a.nul[4] + c), __ldg(a.nul[7] + c), __ldg(a.nul[10] + c)};
    double len = a.uni[0], wid = a.uni[1], spr = a.uni[2], dmp = a.uni[3];
    if constexpr (HET) {
        len = __ldg(a.prm[0] + c); wid = __ldg(a.prm[1] + c);
        spr = __ldg(a.prm[2] + c); dmp = __ldg(a.prm[3] + c);
    }
    const Prm q = make_prm(len, wid, spr, dmp);
    const double g2 = 2.0 * __ldg(a.gcost + c / a.feet);
    const double sF = g2 * a.wf, sT = g2 * a.wt;

    // ---- forward sweep: poses of the segment starts
    const int nseg = (H + S - 1) / S;
    const int tl = (nseg - 1) * S;   // first step of the last segment
    for (int t = 0; t < tl; ++t) {
        if ((t & (S - 1)) == 0) {
            double* k = a.tape + static_cast<long long>(t / S) * 12 * N + c;
            __stcg(k, s.p.x); __stcg(k + N, s.p.y); __stcg(k + 2 * N, s.p.z);
            __stcg(k + 3 * N, s.c0.x); __stcg(k + 4 * N, s.c0.y); __stcg(k + 5 * N, s.c0.z);
            __stcg(k + 6 * N, s.c1.x); __stcg(k + 7 * N, s.c1.y); __stcg(k + 8 * N, s.c1.z);
            __stcg(k + 9 * N, s.c2.x); __stcg(k + 10 * N, s.c2.y); __stcg(k + 11 * N, s.c2.z);
        }
        ptx::cp_async_wait<S - 1>();
        V3 v, w;
        twist(t & (S - 1), v, w);
        kin_euler_step<BAUM>(s, v, w, a.half_rho, a.dT);
        if (t + S < H) stage(t + S, (t + S) & (S - 1));   // the slot just consumed
        ptx::cp_async_commit();
    }
    // the ring now holds the last segment, step tl + j in slot j

    // ---- reverse sweep
    Pose gs{};               // adjoint of the pose
    V3 gp0{}, gn1{}, gn2{};  // null pose
    double gL = 0.0, gW = 0.0, gk = 0.0, gb = 0.0;
    const V3 rf{a.ref[0], a.ref[1], a.ref[2]}, rt{a.ref[3], a.ref[4], a.ref[5]};
    int flip = 0;            // sigma_k(j) = flip ? S-1-j : j
    for (int k = nseg - 1; k >= 0; --k) {
        const int t0 = k * S;
        const int n = min(S, H - t0);
        ptx::cp_async_wait<0>();
        if (k != nseg - 1) {
            const double* ck = a.tape + static_cast<long long>(k) * 12 * N + c;
            s.p = V3{__ldcg(ck), __ldcg(ck + N), __ldcg(ck + 2 * N)};
            s.c0 = V3{__ldcg(ck + 3 * N), __ldcg(ck + 4 * N), __ldcg(ck + 5 * N)};
            s.c1 = V3{__ldcg(ck + 6 * N), __ldcg(ck + 7 * N), __ldcg(ck + 8 * N)};
            s.c2 = V3{__ldcg(ck + 9 * N), __ldcg(ck + 10 * N), __ldcg(ck + 11 * N)};
        }
        for (int j = 0; j < n; ++j) {
            double* o = poses + j * 12 * kWarp + lane;
            o[0] = s.p.x; o[kWarp] = s.p.y; o[2 * kWarp] = s.p.z;
            o[3 * kWarp] = s.c0.x; o[4 * kWarp] = s.c0.y; o[5 * kWarp] = s.c0.z;
            o[6 * kWarp] = s.c1.x; o[7 * kWarp] = s.c1.y; o[8 * kWarp] = s.c1.z;
            o[9 * kWarp] = s.c2.x; o[10 * kWarp] = s.c2.y; o[11 * kWarp] = s.c2.z;
            if (j + 1 < n) {
                V3 v, w;
                twist(flip ? S - 1 - j : j, v, w);
                kin_euler_step<BAUM>(s, v, w, a.half_rho, a.dT);
            }
        }
        // slot sigma_k(j) takes step (k-1)S + S-1-j of the previous segment once step kS + j is done;
        // the slots this (last, short) segment does not use take theirs now
        if (k > 0)
            for (int j = n; j < S; ++j) stage(t0 - 1 - j, flip ? S - 1 - j : j);
        for (int j = n - 1; j >= 0; --j) {
            const int t = t0 + j;
            const int slot = flip ? S - 1 - j : j;
            V3 v, w;
            twist(slot, v, w);
            if (k > 0) stage(t0 - 1 - j, slot);
            const double* o = poses + j * 12 * kWarp + lane;
            Pose ps;
            ps.p = V3{o[0], o[kWarp], o[2 * kWarp]};
            ps.c0 = V3{o[3 * kWarp], o[4 * kWarp], o[5 * kWarp]};
            ps.c1 = V3{o[6 * kWarp], o[7 * kWarp], o[8 * kWarp]};
            ps.c2 = V3{o[9 * kWarp], o[10 * kWarp], o[11 * kWarp]};

            State st;
            st.v = v; st.w = w; st.p = ps.p; st.p0 = p0;
            st.e1 = ps.c0; st.e2 = ps.c1;
            st.R02 = ps.c2.x; st.R12 = ps.c2.y; st.R22 = ps.c2.z;
            st.n1 = n1; st.n2 = n2;
            Result r;
            eval_contact<M_WRENCH>(st, q, r);
            const V3 gF = sF * (r.force - rf), gT = sT * (r.torque - rt);
            VjpOut g;
            vjp_wrench<W>(st, q, len, wid, gF, gT, g);

            const bool last = t == H - 1;   // the step after it does not enter the cost
            V3 gv{}, gw{};
            if constexpr (kTw) gv = g.v, gw = g.w;
            if constexpr (kAdj) {
                if (last) {
                    gs.p = g.p;
                    gs.c0 = g.e1;
                    gs.c1 = g.e2;
                    gs.c2 = V3{0.0, 0.0, g.R22};
                } else {
                    V3 ev{}, ew{};
                    kin_euler_step_vjp<BAUM, kTw>(ps, w, a.half_rho, a.dT, gs, ev, ew);
                    if constexpr (kTw) gv = add_rn(ev, g.v), gw = add_rn(ew, g.w);
                    gs.p = add_rn(gs.p, g.p);
                    gs.c0 = add_rn(gs.c0, g.e1);
                    gs.c1 = add_rn(gs.c1, g.e2);
                    gs.c2.z = __dadd_rn(gs.c2.z, g.R22);
                }
            }
            if constexpr (kTw) {
                const long long i = static_cast<long long>(t) * N + c;
                __stcs(a.gtw[0] + i, gv.x); __stcs(a.gtw[1] + i, gv.y); __stcs(a.gtw[2] + i, gv.z);
                __stcs(a.gtw[3] + i, gw.x); __stcs(a.gtw[4] + i, gw.y); __stcs(a.gtw[5] + i, gw.z);
            }
            if constexpr ((GROUPS & G_NULL) != 0) {
                if (last) gp0 = g.p0, gn1 = g.n1, gn2 = g.n2;
                else gp0 = add_rn(gp0, g.p0), gn1 = add_rn(gn1, g.n1), gn2 = add_rn(gn2, g.n2);
            }
            if constexpr ((GROUPS & G_PARAMS) != 0) {
                if (last) gL = g.L, gW = g.W, gk = g.k, gb = g.b;
                else gL = __dadd_rn(gL, g.L), gW = __dadd_rn(gW, g.W), gk = __dadd_rn(gk, g.k), gb = __dadd_rn(gb, g.b);
            }
        }
        ptx::cp_async_commit();
        flip ^= 1;
    }

    if constexpr ((GROUPS & G_POSE) != 0) {
        a.gpos[0][c] = gs.p.x; a.gpos[1][c] = gs.p.y; a.gpos[2][c] = gs.p.z;
        a.grot[0][c] = gs.c0.x; a.grot[1][c] = gs.c1.x; a.grot[2][c] = gs.c2.x;
        a.grot[3][c] = gs.c0.y; a.grot[4][c] = gs.c1.y; a.grot[5][c] = gs.c2.y;
        a.grot[6][c] = gs.c0.z; a.grot[7][c] = gs.c1.z; a.grot[8][c] = gs.c2.z;
    }
    if constexpr ((GROUPS & G_NULL) != 0) {
        a.gnul[0][c] = gp0.x; a.gnul[1][c] = gp0.y; a.gnul[2][c] = gp0.z;
        a.gnul[3][c] = gn1.x; a.gnul[4][c] = gn2.x; a.gnul[5][c] = 0.0;
        a.gnul[6][c] = gn1.y; a.gnul[7][c] = gn2.y; a.gnul[8][c] = 0.0;
        a.gnul[9][c] = gn1.z; a.gnul[10][c] = gn2.z; a.gnul[11][c] = 0.0;
    }
    if constexpr ((GROUPS & G_PARAMS) != 0) {
        a.gprm[0][c] = gL; a.gprm[1][c] = gW; a.gprm[2][c] = gk; a.gprm[3][c] = gb;
    }
}

// ------------------------------------------------------------------------------------------------
// Warp-specialised rollout for SMALL batches, cost only.
//
// A sampling-MPC batch of configs[2] size has 8 192 chains: 256 warps for 592 warp schedulers, and
// every warp walks 100 dependent steps -- latency, not throughput, sets the time.  Only the pose
// integration is inherently sequential.  So a CTA shares one 32-chain tile: warp 0 (producer)
// integrates the pose and publishes it per step into a shared-memory ring, C consumer warps
// evaluate the contact wrench and the cost of the steps t = k (mod C); no work is duplicated (the
// `split` form above lets every warp integrate everything).  The producer's instruction stream is
// the critical path (100 dependent steps whatever the batch size), so everything that is not the
// pose recurrence leaves it:
//   * the twists of step t+1 are lifted out of the cp.async ring into registers while step t is
//     integrated (the 29-cycle shared-memory latency is off the chain);
//   * a stage holds only the pose (p, e1, e2, R22: 10 doubles per lane, five 128-bit stores); the
//     consumers fetch the twist of their own steps straight from global memory, one step ahead;
//   * stages are handed over in GROUPS of C (one stage per consumer): the producer waits on ONE
//     `empty` barrier per C steps (an mbarrier try_wait costs ~90 cycles even when it succeeds) and
//     signals ONE `full` barrier per group; consumer k evaluates step g*C + k of every group g;
//   * C consumer warps (3, 5 or 7) keep up with the leaner producer.
// Works with and without the Baumgarte term.  chain_cost[chain*C + k] = consumer k's partial cost;
// the reduction kernel sums a rollout's feet*C partials in index order (deterministic).
// ------------------------------------------------------------------------------------------------

constexpr int kWs2Groups = 3;               // stage groups in flight
constexpr int kWs2StageDoubles = 10 * kWarp;

template <int C>
struct Ws2Cfg {
    static constexpr int kStages = kWs2Groups * C;
    static constexpr int kThreads = kWarp * (C + 1);
    static constexpr int kSmemBytes = kRolloutRingBytes + kStages * kWs2StageDoubles * 8 + 2 * kWs2Groups * 8 + 64;
};

template <bool HET, bool BAUM, int C>
__global__ void __launch_bounds__(kWarp * (C + 1))
ccm_rollout_ws2_kernel(const __grid_constant__ RolloutArgs a)
{
    constexpr int D = kRolloutDepth;
    constexpr int S = Ws2Cfg<C>::kStages;
    constexpr int NG = kWs2Groups;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long wbase = static_cast<long long>(blockIdx.x) * kWarp;
    const long long c = wbase + lane;
    const bool on = c < a.chains;
    const int H = a.horizon;

    double* ring = reinterpret_cast<double*>(smem_raw);                       // producer's twist ring
    double* stages = ring + D * 6 * kWarp;                                    // [S][10][32]
    const uint32_t full0 = ptx::smem_addr(stages + S * kWs2StageDoubles);     // NG barriers, 1 arrival
    const uint32_t empty0 = full0 + 8 * NG;                                   // NG barriers, C arrivals
    if (threadIdx.x == 0) {
        for (int g = 0; g < NG; ++g) {
            ptx::mbar_init(full0 + 8 * g, 1);
            ptx::mbar_init(empty0 + 8 * g, C);
        }
        ptx::fence_mbar_init();
    }
    __syncthreads();

    if (warp == 0) {
        // ---------------- producer: the pose recurrence and nothing else -------------------------
        const uint32_t ring_s = ptx::smem_addr(ring) + static_cast<uint32_t>(lane) * 8u;
        const double* src[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) src[j] = a.tw[j] + c;
#pragma unroll
        for (int t = 0; t < D; ++t) {
            if (on && t < H) {
                const uint32_t dst = ring_s + static_cast<uint32_t>(t * 6 * kWarp * 8);
#pragma unroll
                for (int j = 0; j < 6; ++j) ptx::cp_async8(dst + j * kWarp * 8, src[j] + static_cast<long long>(t) * a.chains);
            }
            ptx::cp_async_commit();
        }
#pragma unroll
        for (int j = 0; j < 6; ++j) src[j] += static_cast<long long>(D) * a.chains;   // step t + D
        Pose s{};
        if (on) {
            s.p = V3{__ldg(a.pos0[0] + c), __ldg(a.pos0[1] + c), __ldg(a.pos0[2] + c)};
            s.c0 = V3{__ldg(a.rot0[0] + c), __ldg(a.rot0[3] + c), __ldg(a.rot0[6] + c)};
            s.c1 = V3{__ldg(a.rot0[1] + c), __ldg(a.rot0[4] + c), __ldg(a.rot0[7] + c)};
            s.c2 = V3{__ldg(a.rot0[2] + c), __ldg(a.rot0[5] + c), __ldg(a.rot0[8] + c)};
        }
        // twist of step 0 into registers
        ptx::cp_async_wait<D - 1>();
        V3 vn{}, wn{};
        if (on) {
            const double* r = ring + lane;
            vn = V3{r[0], r[kWarp], r[2 * kWarp]};
            wn = V3{r[3 * kWarp], r[4 * kWarp], r[5 * kWarp]};
        }
        int slot = 0;               // twist ring slot of step t
        int st = 0;                 // stage of step t
        int gi = 0, g = 0;          // position inside the group, group slot
        uint32_t empty_parity = 0;
        bool wrapped = false;
        for (int t = 0; t < H; ++t) {
            const V3 v = vn, w = wn;
            // the twist of step t + 1 (its copy was issued D - 1 steps ago): in flight while step t is integrated
            ptx::cp_async_wait<D - 2>();
            const int nslot = (slot + 1) & (D - 1);
            if (on) {
                const double* r = ring + nslot * 6 * kWarp + lane;
                vn = V3{r[0], r[kWarp], r[2 * kWarp]};
                wn = V3{r[3 * kWarp], r[4 * kWarp], r[5 * kWarp]};
            }
            if (gi == 0 && wrapped) ptx::mbar_wait(empty0 + 8 * g, empty_parity);   // the group's stages are free
            double2* o = reinterpret_cast<double2*>(stages + st * kWs2StageDoubles) + lane;
            o[0 * kWarp] = make_double2(s.p.x, s.p.y);
            o[1 * kWarp] = make_double2(s.p.z, s.c0.x);
            o[2 * kWarp] = make_double2(s.c0.y, s.c0.z);
            o[3 * kWarp] = make_double2(s.c1.x, s.c1.y);
            o[4 * kWarp] = make_double2(s.c1.z, s.c2.z);
            kin_euler_step<BAUM>(s, v, w, a.half_rho, a.dT);
            if (++gi == C || t == H - 1) {   // the group is complete: hand it over
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(full0 + 8 * g);
                gi = 0;
                if (++g == NG) {
                    g = 0;
                    empty_parity = wrapped ? (empty_parity ^ 1u) : 0u;
                    wrapped = true;
                }
            }
            // refill the ring slot of step t (read one iteration ago) with step t + D
            if (on && t + D < H) {
                const uint32_t dst = ring_s + static_cast<uint32_t>(slot * 6 * kWarp * 8);
#pragma unroll
                for (int j = 0; j < 6; ++j) ptx::cp_async8(dst + j * kWarp * 8, src[j]);
            }
            ptx::cp_async_commit();
#pragma unroll
            for (int j = 0; j < 6; ++j) src[j] += a.chains;
            slot = nslot;
            if (++st == S) st = 0;
        }
        if (on && a.write_final) {
            a.pos_out[0][c] = s.p.x; a.pos_out[1][c] = s.p.y; a.pos_out[2][c] = s.p.z;
            a.rot_out[0][c] = s.c0.x; a.rot_out[1][c] = s.c1.x; a.rot_out[2][c] = s.c2.x;
            a.rot_out[3][c] = s.c0.y; a.rot_out[4][c] = s.c1.y; a.rot_out[5][c] = s.c2.y;
            a.rot_out[6][c] = s.c0.z; a.rot_out[7][c] = s.c1.z; a.rot_out[8][c] = s.c2.z;
        }
        ptx::cp_async_wait<0>();
    } else {
        // ---------------- consumer k: contact wrench + cost of the steps g*C + k -----------------
        const int k = warp - 1;
        V3 p0{}, n1{}, n2{};
        Prm q = a.uni;
        if (on) {
            p0 = V3{__ldg(a.nul[0] + c), __ldg(a.nul[1] + c), __ldg(a.nul[2] + c)};
            n1 = V3{__ldg(a.nul[3] + c), __ldg(a.nul[6] + c), __ldg(a.nul[9] + c)};
            n2 = V3{__ldg(a.nul[4] + c), __ldg(a.nul[7] + c), __ldg(a.nul[10] + c)};
            if constexpr (HET)
                q = make_prm(__ldg(a.prm[0] + c), __ldg(a.prm[1] + c), __ldg(a.prm[2] + c),
                             __ldg(a.prm[3] + c));
        }
        // the twists of this consumer's own steps come straight from global memory, one step ahead
        const long long tstride = static_cast<long long>(C) * a.chains;
        long long ti = static_cast<long long>(k) * a.chains + c;
        V3 vn{}, wn{};
        if (on && k < H) {
            vn = V3{__ldg(a.tw[0] + ti), __ldg(a.tw[1] + ti), __ldg(a.tw[2] + ti)};
            wn = V3{__ldg(a.tw[3] + ti), __ldg(a.tw[4] + ti), __ldg(a.tw[5] + ti)};
        }
        double acc = 0.0;
        int g = 0;
        uint32_t parity = 0;
        const double2* stage_k = reinterpret_cast<const double2*>(stages + k * kWs2StageDoubles) + lane;
        for (int t = k; t < H; t += C) {
            State x;
            x.v = vn;
            x.w = wn;
            ti += tstride;
            if (on && t + C < H) {
                vn = V3{__ldg(a.tw[0] + ti), __ldg(a.tw[1] + ti), __ldg(a.tw[2] + ti)};
                wn = V3{__ldg(a.tw[3] + ti), __ldg(a.tw[4] + ti), __ldg(a.tw[5] + ti)};
            }
            ptx::mbar_wait(full0 + 8 * g, parity);
            const double2* in = stage_k + g * (C * kWs2StageDoubles / 2);
            const double2 a0 = in[0 * kWarp], a1 = in[1 * kWarp], a2 = in[2 * kWarp], a3 = in[3 * kWarp],
                          a4 = in[4 * kWarp];
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(empty0 + 8 * g);   // one of the C arrivals that free the group
            x.p = V3{a0.x, a0.y, a1.x};
            x.e1 = V3{a1.y, a2.x, a2.y};
            x.e2 = V3{a3.x, a3.y, a4.x};
            x.R02 = 0.0; x.R12 = 0.0;
            x.R22 = a4.y;
            x.p0 = p0; x.n1 = n1; x.n2 = n2;
            Result r;
            eval_contact<M_WRENCH>(x, q, r);
            if (on) {
                const V3 df = r.force - V3{a.ref[0], a.ref[1], a.ref[2]};
                const V3 dt = r.torque - V3{a.ref[3], a.ref[4], a.ref[5]};
                acc = acc + (a.wf * (df.x * df.x + df.y * df.y + df.z * df.z) +
                             a.wt * (dt.x * dt.x + dt.y * dt.y + dt.z * dt.z));
            }
            if (++g == NG) {
                g = 0;
                parity ^= 1u;
            }
        }
        if (on) a.chain_cost[c * C + k] = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// Third form: the same producer / consumer split with the last avoidable work taken off the
// producer and the second launch removed.
//   * Twists arrive by TMA TENSOR copies (cp.async.bulk.tensor.2d, SASS UTMALDG): the six planes are
//     [horizon][chains] tensors, one box = 8 steps x 32 chains (2 KB per plane), two boxes in
//     flight; one elected lane issues six copies per EIGHT steps and the warp waits on one
//     mbarrier per box.  The per-lane cp.async ring of the second form cost ~50 instructions per
//     step on the critical warp (six 64-bit pointer increments, six LDGSTS, the commit/wait
//     bookkeeping; ncu: 215 instructions and 774 cycles per step with the Baumgarte term).  Rows
//     past the horizon and columns past the last chain are zero-filled by the hardware.
//   * The step loop is unrolled over a box, so ring slots and shared-memory offsets are immediates.
//   * The reduction is fused: consumers leave their partial costs in shared memory, warp 0 sums each
//     rollout's feet*C partials in index order (the order of ccm_cost_reduce_kernel: bit-identical),
//     arg-mins over the tile, and the last CTA to finish combines the CTAs' pairs and -- if enabled
//     -- runs the NVLink peer exchange.  One launch per MPC step instead of two.
// Needs: 32 % feet == 0 (no rollout straddles a tile), chains even and plane bases 16-byte aligned
// (TMA global-stride rule); otherwise the second form + ccm_cost_reduce_kernel run.
// ------------------------------------------------------------------------------------------------

constexpr int kWs3BoxSteps = 8;
constexpr int kWs3Boxes = 2;
constexpr int kWs3BoxBytes = 6 * kWs3BoxSteps * kWarp * 8;   // 12 288 per box (six planes)

template <int C>
struct Ws3Cfg {
    static constexpr int kStages = kWs2Groups * C;
    static constexpr int kThreads = kWarp * (C + 1);
    static constexpr int kBarBytes = 128;
    static constexpr int kSmemBytes = kWs3Boxes * kWs3BoxBytes + kStages * kWs2StageDoubles * 8 + kBarBytes +
                                      kWarp * C * 8;
};

namespace ptx {
// 2-D tiled tensor copy global -> shared::cta, completion in bytes on an mbarrier (SASS: UTMALDG)
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* map, int c0, int c1, uint32_t bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
// bring a tensor map (kernel parameter) into the descriptor cache ahead of its first use
__device__ __forceinline__ void prefetch_tensormap(const void* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
}  // namespace ptx

template <bool HET, bool BAUM, int C>
__global__ void __launch_bounds__(kWarp * (C + 1))
ccm_rollout_ws3_kernel(const __grid_constant__ RolloutArgs a)
{
    constexpr int S = Ws3Cfg<C>::kStages;
    constexpr int NG = kWs2Groups;
    constexpr int BS = kWs3BoxSteps;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long wbase = static_cast<long long>(blockIdx.x) * kWarp;
    const long long c = wbase + lane;
    const bool on = c < a.chains;
    const int H = a.horizon;

    double* twbuf = reinterpret_cast<double*>(smem_raw);                              // [box][plane][step][lane]
    double* stages = twbuf + kWs3Boxes * kWs3BoxBytes / 8;                            // [S][10][32]
    const uint32_t bars = ptx::smem_addr(stages + S * kWs2StageDoubles);
    const uint32_t twfull0 = bars;                 // kWs3Boxes barriers: a box has landed
    const uint32_t full0 = bars + 8 * kWs3Boxes;   // NG barriers, 1 arrival: a stage group is written
    const uint32_t empty0 = full0 + 8 * NG;        // NG barriers, C arrivals: a stage group is consumed
    double* cst = stages + S * kWs2StageDoubles + Ws3Cfg<C>::kBarBytes / 8;           // [32][C] partial costs
    if (threadIdx.x == 0) {
        for (int b = 0; b < kWs3Boxes; ++b) ptx::mbar_init(twfull0 + 8 * b, 1);
        for (int g = 0; g < NG; ++g) {
            ptx::mbar_init(full0 + 8 * g, 1);
            ptx::mbar_init(empty0 + 8 * g, C);
        }
        ptx::fence_mbar_init();
    }
    __syncthreads();

    if (warp == 0) {
        // ---------------- producer: the pose recurrence and nothing else -------------------------
        const int nbox = (H + BS - 1) / BS;
        auto load_box = [&](int b) {   // lane 0: the six planes' box b into buffer b % kWs3Boxes
            const int buf = b & (kWs3Boxes - 1);
            const uint32_t bar = twfull0 + 8 * buf;
            const uint32_t dst = ptx::smem_addr(twbuf) + buf * kWs3BoxBytes;
            ptx::mbar_arrive_expect_tx(bar, kWs3BoxBytes);
#pragma unroll
            for (int j = 0; j < 6; ++j)
                ptx::tma_load_2d(dst + j * (BS * kWarp * 8), &a.twmap[j], static_cast<int>(wbase), b * BS, bar);
        };
        if (lane == 0) {
#pragma unroll
            for (int b = 0; b < kWs3Boxes; ++b)
                if (b < nbox) load_box(b);
        }
        Pose s{};
        if (on) {
            s.p = V3{__ldg(a.pos0[0] + c), __ldg(a.pos0[1] + c), __ldg(a.pos0[2] + c)};
            s.c0 = V3{__ldg(a.rot0[0] + c), __ldg(a.rot0[3] + c), __ldg(a.rot0[6] + c)};
            s.c1 = V3{__ldg(a.rot0[1] + c), __ldg(a.rot0[4] + c), __ldg(a.rot0[7] + c)};
            s.c2 = V3{__ldg(a.rot0[2] + c), __ldg(a.rot0[5] + c), __ldg(a.rot0[8] + c)};
        }
        const double half_rho = a.half_rho, dT = a.dT;
        int st = 0;                 // stage of step t
        int gi = 0, g = 0;          // position inside the group, group slot
        uint32_t empty_parity = 0;
        bool wrapped = false;
        uint32_t box_parity = 0;    // parity of the box buffers' current use (both buffers flip together)
        for (int b = 0; b < nbox; ++b) {
            const int buf = b & (kWs3Boxes - 1);
            ptx::mbar_wait(twfull0 + 8 * buf, box_parity);
            if (buf == kWs3Boxes - 1) box_parity ^= 1u;
            const double* tw = twbuf + buf * (kWs3BoxBytes / 8) + lane;
            const int steps = min(BS, H - b * BS);
            V3 vn{tw[0], tw[BS * kWarp], tw[2 * BS * kWarp]};
            V3 wn{tw[3 * BS * kWarp], tw[4 * BS * kWarp], tw[5 * BS * kWarp]};
#pragma unroll
            for (int q = 0; q < BS; ++q) {
                if (q < steps) {
                    const V3 v = vn, w = wn;
                    if (q + 1 < BS) {   // next step's twist: in flight while this step is integrated
                        const double* r = tw + (q + 1) * kWarp;
                        vn = V3{r[0], r[BS * kWarp], r[2 * BS * kWarp]};
                        wn = V3{r[3 * BS * kWarp], r[4 * BS * kWarp], r[5 * BS * kWarp]};
                    }
                    if (gi == 0 && wrapped) ptx::mbar_wait(empty0 + 8 * g, empty_parity);   // the group's stages are free
                    double2* o = reinterpret_cast<double2*>(stages + st * kWs2StageDoubles) + lane;
                    o[0 * kWarp] = make_double2(s.p.x, s.p.y);
                    o[1 * kWarp] = make_double2(s.p.z, s.c0.x);
                    o[2 * kWarp] = make_double2(s.c0.y, s.c0.z);
                    o[3 * kWarp] = make_double2(s.c1.x, s.c1.y);
                    o[4 * kWarp] = make_double2(s.c1.z, s.c2.z);
                    kin_euler_step<BAUM>(s, v, w, half_rho, dT);
                    if (++gi == C || b * BS + q == H - 1) {   // the group is complete: hand it over
                        __syncwarp();
                        if (lane == 0) ptx::mbar_arrive(full0 + 8 * g);
                        gi = 0;
                        if (++g == NG) {
                            g = 0;
                            empty_parity = wrapped ? (empty_parity ^ 1u) : 0u;
                            wrapped = true;
                        }
                    }
                    if (++st == S) st = 0;
                }
            }
            // every lane holds the box's last twist in registers: the buffer may be refilled
            __syncwarp();
            if (lane == 0 && b + kWs3Boxes < nbox) {
                ptx::fence_async_smem();
                load_box(b + kWs3Boxes);
            }
        }
        if (on && a.write_final) {
            a.pos_out[0][c] = s.p.x; a.pos_out[1][c] = s.p.y; a.pos_out[2][c] = s.p.z;
            a.rot_out[0][c] = s.c0.x; a.rot_out[1][c] = s.c1.x; a.rot_out[2][c] = s.c2.x;
            a.rot_out[3][c] = s.c0.y; a.rot_out[4][c] = s.c1.y; a.rot_out[5][c] = s.c2.y;
            a.rot_out[6][c] = s.c0.z; a.rot_out[7][c] = s.c1.z; a.rot_out[8][c] = s.c2.z;
        }
    } else {
        // ---------------- consumer k: contact wrench + cost of the steps g*C + k -----------------
        const int k = warp - 1;
        V3 p0{}, n1{}, n2{};
        Prm q = a.uni;
        if (on) {
            p0 = V3{__ldg(a.nul[0] + c), __ldg(a.nul[1] + c), __ldg(a.nul[2] + c)};
            n1 = V3{__ldg(a.nul[3] + c), __ldg(a.nul[6] + c), __ldg(a.nul[9] + c)};
            n2 = V3{__ldg(a.nul[4] + c), __ldg(a.nul[7] + c), __ldg(a.nul[10] + c)};
            if constexpr (HET)
                q = make_prm(__ldg(a.prm[0] + c), __ldg(a.prm[1] + c), __ldg(a.prm[2] + c),
                             __ldg(a.prm[3] + c));
        }
        // the twists of this consumer's own steps come straight from global memory, one step ahead
        const long long tstride = static_cast<long long>(C) * a.chains;
        long long ti = static_cast<long long>(k) * a.chains + c;
        V3 vn{}, wn{};
        if (on && k < H) {
            vn = V3{__ldg(a.tw[0] + ti), __ldg(a.tw[1] + ti), __ldg(a.tw[2] + ti)};
            wn = V3{__ldg(a.tw[3] + ti), __ldg(a.tw[4] + ti), __ldg(a.tw[5] + ti)};
        }
        double acc = 0.0;
        int g = 0;
        uint32_t parity = 0;
        const double2* stage_k = reinterpret_cast<const double2*>(stages + k * kWs2StageDoubles) + lane;
        for (int t = k; t < H; t += C) {
            State x;
            x.v = vn;
            x.w = wn;
            ti += tstride;
            if (on && t + C < H) {
                vn = V3{__ldg(a.tw[0] + ti), __ldg(a.tw[1] + ti), __ldg(a.tw[2] + ti)};
                wn = V3{__ldg(a.tw[3] + ti), __ldg(a.tw[4] + ti), __ldg(a.tw[5] + ti)};
            }
            ptx::mbar_wait(full0 + 8 * g, parity);
            const double2* in = stage_k + g * (C * kWs2StageDoubles / 2);
            const double2 a0 = in[0 * kWarp], a1 = in[1 * kWarp], a2 = in[2 * kWarp], a3 = in[3 * kWarp],
                          a4 = in[4 * kWarp];
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(empty0 + 8 * g);   // one of the C arrivals that free the group
            x.p = V3{a0.x, a0.y, a1.x};
            x.e1 = V3{a1.y, a2.x, a2.y};
            x.e2 = V3{a3.x, a3.y, a4.x};
            x.R02 = 0.0; x.R12 = 0.0;
            x.R22 = a4.y;
            x.p0 = p0; x.n1 = n1; x.n2 = n2;
            Result r;
            eval_contact<M_WRENCH>(x, q, r);
            if (on) {
                const V3 df = r.force - V3{a.ref[0], a.ref[1], a.ref[2]};
                const V3 dt = r.torque - V3{a.ref[3], a.ref[4], a.ref[5]};
                acc = acc + (a.wf * (df.x * df.x + df.y * df.y + df.z * df.z) +
                             a.wt * (dt.x * dt.x + dt.y * dt.y + dt.z * dt.z));
            }
            if (++g == NG) {
                g = 0;
                parity ^= 1u;
            }
        }
        cst[lane * C + k] = acc;    // chains past the end: 0, never read
    }

    // ---------------- fused reduction: rollout costs of this tile, arg-min, last CTA combines -----
    __syncthreads();
    if (warp != 0) return;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    CostIdx mine{inf, 0x7fffffffffffffffLL};
    {
        const int feet = a.feet;
        const long long ro = wbase / feet + lane;          // 32 % feet == 0: tiles hold whole rollouts
        if (lane < kWarp / feet && ro < a.n_rollouts) {
            const double* p = cst + lane * feet * C;
            double sum = 0.0;
            for (int j = 0; j < feet * C; ++j) sum += p[j];
            if (a.cost) a.cost[ro] = sum;
            mine.cost = sum;
            mine.idx = a.index_base + ro;
            if (!(sum == sum)) mine = CostIdx{inf, 0x7fffffffffffffffLL};   // NaN never wins
        }
    }
    mine = warp_best(mine);
    if (lane == 0) {
        a.block_best[blockIdx.x] = mine;
        __threadfence();
        const unsigned int done = atomicAdd(a.counter, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncwarp();
    if (!s_last) return;
    __threadfence();
    CostIdx b{inf, 0x7fffffffffffffffLL};
    for (unsigned int j = lane; j < gridDim.x; j += kWarp) {
        CostIdx cand;
        cand.cost = *reinterpret_cast<volatile double*>(&a.block_best[j].cost);
        cand.idx = *reinterpret_cast<volatile long long*>(&a.block_best[j].idx);
        if (better(cand.cost, cand.idx, b.cost, b.idx)) b = cand;
    }
    b = warp_best(b);
    if (b.idx == 0x7fffffffffffffffLL) b.idx = -1;  // nothing comparable (empty / all NaN)
    if (lane == 0) {
        *a.best = b;
        *a.counter = 0u;
    }
    if (a.p2p.nranks > 0) {   // fused collective: this rank's pair goes straight to the peers' mailboxes
        const CostIdx gbest = p2p_exchange_warp(a.p2p, b, lane);
        if (lane == 0) *a.p2p.out = gbest;
    }
}

// ------------------------------------------------------------------------------------------------
// Fourth form: the pose recurrence itself is spread over LANES.
//
// ncu on the second form showed what bounds a small batch: the lone producer warp issues one
// instruction every ~3.6 cycles (a single warp per scheduler: every dependent or same-pipe
// instruction waits), so the per-step time is its instruction count -- 215 instructions, 774 cycles
// with the Baumgarte term.  The third form cut that to ~117.  Here FOUR lanes share a chain: lanes
// 0-2 own one column of R each, lane 3 owns the position; the columns' updates are independent
// given w (three lanes do in parallel what one lane did in sequence), and the Baumgarte term,
// which couples the columns, gets the two other columns by warp shuffles (k_j = c_{j+1} x c_{j+2}
// is cyclic, so every lane runs the same code) and dT rho/2 / det R from lane 0 (the one value
// every other kernel uses, so results stay bit-identical to them).  A 32-chain tile now has four
// producer warps of 8 chains; per lane and step ~9 (rho = 0) or ~30 (rho != 0) FP64 instructions
// instead of 30 / 75.  Twists by TMA tensor copies, stage hand-over in groups, C consumer warps
// and the fused reduction exactly as in the third form.
// ------------------------------------------------------------------------------------------------

constexpr int kWs4Producers = 4;
constexpr int kWs4StageDoubles = 16 * kWarp;   // 8 double2 slots x 32 chains: p.xy p.z_ c0.xy c0.z_ c1.xy c1.z_ c2.xy c2.z_

template <int C>
struct Ws4Cfg {
    static constexpr int kStages = kWs2Groups * C;
    static constexpr int kThreads = kWarp * (kWs4Producers + C);
    static constexpr int kBarBytes = 128;
    static constexpr int kSmemBytes = kWs3Boxes * kWs3BoxBytes + kStages * kWs4StageDoubles * 8 + kBarBytes +
                                      kWarp * C * 8;
};

__device__ __forceinline__ V3 shfl3(const V3& a, int src)
{
    return V3{__shfl_sync(0xffffffffu, a.x, src), __shfl_sync(0xffffffffu, a.y, src),
              __shfl_sync(0xffffffffu, a.z, src)};
}

template <bool HET, bool BAUM, int C>
__global__ void __launch_bounds__(kWarp * (kWs4Producers + C))
ccm_rollout_ws4_kernel(const __grid_constant__ RolloutArgs a)
{
    constexpr int NP = kWs4Producers;
    constexpr int S = Ws4Cfg<C>::kStages;
    constexpr int NG = kWs2Groups;
    constexpr int BS = kWs3BoxSteps;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long wbase = static_cast<long long>(blockIdx.x) * kWarp;
    const int H = a.horizon;

    double* twbuf = reinterpret_cast<double*>(smem_raw);                              // [box][plane][step][chain]
    double* stages = twbuf + kWs3Boxes * kWs3BoxBytes / 8;                            // [S][8 slots][32] double2
    const uint32_t bars = ptx::smem_addr(stages + S * kWs4StageDoubles);
    const uint32_t twfull0 = bars;                        // a box has landed (TMA bytes)
    const uint32_t twempty0 = twfull0 + 8 * kWs3Boxes;    // NP arrivals: every producer warp has read the box
    const uint32_t full0 = twempty0 + 8 * kWs3Boxes;      // NP arrivals: a stage group is written
    const uint32_t empty0 = full0 + 8 * NG;               // C arrivals: a stage group is consumed
    double* cst = stages + S * kWs4StageDoubles + Ws4Cfg<C>::kBarBytes / 8;           // [32][C] partial costs
    if (threadIdx.x == 0) {
        for (int b = 0; b < kWs3Boxes; ++b) {
            ptx::mbar_init(twfull0 + 8 * b, 1);
            ptx::mbar_init(twempty0 + 8 * b, NP);
        }
        for (int g = 0; g < NG; ++g) {
            ptx::mbar_init(full0 + 8 * g, NP);
            ptx::mbar_init(empty0 + 8 * g, C);
        }
        ptx::fence_mbar_init();
    }
    __syncthreads();

    if (warp < NP) {
        // ---------------- producers: lane = 4 * (chain in warp) + part; part 0-2 = column of R, 3 = position
        const int part = lane & 3;
        const int ct = warp * 8 + (lane >> 2);            // chain inside the tile
        const long long c = wbase + ct;
        const bool on = c < a.chains;
        const bool is_p = part == 3;
        const int nbox = (H + BS - 1) / BS;
        auto load_box = [&](int b) {   // one thread: the six planes' box b into buffer b % kWs3Boxes
            const int buf = b & (kWs3Boxes - 1);
            const uint32_t bar = twfull0 + 8 * buf;
            const uint32_t dst = ptx::smem_addr(twbuf) + buf * kWs3BoxBytes;
            ptx::mbar_arrive_expect_tx(bar, kWs3BoxBytes);
#pragma unroll
            for (int j = 0; j < 6; ++j)
                ptx::tma_load_2d(dst + j * (BS * kWarp * 8), &a.twmap[j], static_cast<int>(wbase), b * BS, bar);
        };
        if (threadIdx.x == 0) {
#pragma unroll
            for (int b = 0; b < kWs3Boxes; ++b)
                if (b < nbox) load_box(b);
        }
        // this lane's state vector: a column of R (row-major planes part, 3 + part, 6 + part) or the position
        V3 x{};
        if (on) {
            x = is_p ? V3{__ldg(a.pos0[0] + c), __ldg(a.pos0[1] + c), __ldg(a.pos0[2] + c)}
                     : V3{__ldg(a.rot0[part] + c), __ldg(a.rot0[3 + part] + c), __ldg(a.rot0[6 + part] + c)};
        }
        // the twist half this lane needs: angular (planes 3-5) for a column, linear (0-2) for the position
        const double* twl = twbuf + (is_p ? 0 : 3) * BS * kWarp + ct;
        // the two other columns, cyclically: part j gets c_{j+1} and c_{j+2}; the position lane reads itself
        const int lb = lane & ~3;
        const int srcA = is_p ? lane : lb + (part + 1) % 3, srcB = is_p ? lane : lb + (part + 2) % 3;
        const double dT = a.dT;
        const double alpha = is_p ? 1.0 : kin_alpha(dT, a.half_rho);
        const double dthr = kin_dthr(dT, a.half_rho);
        // stage slots of this lane's vector: p -> 0,1; column j -> 2 + 2j, 3 + 2j
        const int slot0 = is_p ? 0 : 2 + 2 * part;
        int st = 0;
        int gi = 0, g = 0;
        uint32_t empty_parity = 0;
        bool wrapped = false;
        uint32_t box_parity = 0;
        for (int b = 0; b < nbox; ++b) {
            const int buf = b & (kWs3Boxes - 1);
            ptx::mbar_wait(twfull0 + 8 * buf, box_parity);
            const double* tw = twl + buf * (kWs3BoxBytes / 8);
            const int steps = min(BS, H - b * BS);
            V3 un{tw[0], tw[BS * kWarp], tw[2 * BS * kWarp]};
#pragma unroll
            for (int q = 0; q < BS; ++q) {
                if (q < steps) {
                    const V3 u = un;
                    if (q + 1 < BS) {   // next step's twist: in flight while this step is integrated
                        const double* r = tw + (q + 1) * kWarp;
                        un = V3{r[0], r[BS * kWarp], r[2 * BS * kWarp]};
                    }
                    if (gi == 0 && wrapped) ptx::mbar_wait(empty0 + 8 * g, empty_parity);   // the group's stages are free
                    double2* o = reinterpret_cast<double2*>(stages + st * kWs4StageDoubles) + slot0 * kWarp + ct;
                    o[0] = make_double2(x.x, x.y);
                    o[kWarp] = make_double2(x.z, 0.0);
                    // ---- one ForwardEuler step of this lane's vector (kin_euler_step, one column per lane)
                    V3 k{};
                    double beta = 0.0;
                    if constexpr (BAUM) {
                        const V3 ca = shfl3(x, srcA), cb = shfl3(x, srcB);
                        k = cross(ca, cb);                                  // position lane: p x p = 0
                        const double bl = __dmul_rn(dthr, fast_rcp(dot3(x, k)));   // part 0: dT rho/2 / (c0 . (c1 x c2))
                        beta = __shfl_sync(0xffffffffu, bl, lb);            // every kernel uses THAT determinant
                        if (is_p) beta = 0.0;
                    }
                    const V3 xc = cross(u, x);                              // w x c_j
                    const V3 rate = is_p ? u : xc;                          // the position integrates v itself
                    x = kin_col_step<BAUM>(x, rate, k, alpha, beta, dT);
                    if (++gi == C || b * BS + q == H - 1) {   // the group is complete: hand it over
                        __syncwarp();
                        if (lane == 0) ptx::mbar_arrive(full0 + 8 * g);
                        gi = 0;
                        if (++g == NG) {
                            g = 0;
                            empty_parity = wrapped ? (empty_parity ^ 1u) : 0u;
                            wrapped = true;
                        }
                    }
                    if (++st == S) st = 0;
                }
            }
            // this warp holds the box's last twist in registers: release the buffer; thread 0 refills it
            // once all four producer warps have
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(twempty0 + 8 * buf);
            if (threadIdx.x == 0 && b + kWs3Boxes < nbox) {
                ptx::mbar_wait(twempty0 + 8 * buf, box_parity);
                ptx::fence_async_smem();
                load_box(b + kWs3Boxes);
            }
            if (buf == kWs3Boxes - 1) box_parity ^= 1u;
        }
        if (on && a.write_final) {
            if (is_p) {
                a.pos_out[0][c] = x.x; a.pos_out[1][c] = x.y; a.pos_out[2][c] = x.z;
            } else {
                a.rot_out[part][c] = x.x; a.rot_out[3 + part][c] = x.y; a.rot_out[6 + part][c] = x.z;
            }
        }
    } else {
        // ---------------- consumer k: contact wrench + cost of the steps g*C + k -----------------
        const long long c = wbase + lane;
        const bool on = c < a.chains;
        const int k = warp - NP;
        V3 p0{}, n1{}, n2{};
        Prm q = a.uni;
        if (on) {
            p0 = V3{__ldg(a.nul[0] + c), __ldg(a.nul[1] + c), __ldg(a.nul[2] + c)};
            n1 = V3{__ldg(a.nul[3] + c), __ldg(a.nul[6] + c), __ldg(a.nul[9] + c)};
            n2 = V3{__ldg(a.nul[4] + c), __ldg(a.nul[7] + c), __ldg(a.nul[10] + c)};
            if constexpr (HET)
                q = make_prm(__ldg(a.prm[0] + c), __ldg(a.prm[1] + c), __ldg(a.prm[2] + c),
                             __ldg(a.prm[3] + c));
        }
        const long long tstride = static_cast<long long>(C) * a.chains;
        long long ti = static_cast<long long>(k) * a.chains + c;
        V3 vn{}, wn{};
        if (on && k < H) {
            vn = V3{__ldg(a.tw[0] + ti), __ldg(a.tw[1] + ti), __ldg(a.tw[2] + ti)};
            wn = V3{__ldg(a.tw[3] + ti), __ldg(a.tw[4] + ti), __ldg(a.tw[5] + ti)};
        }
        double acc = 0.0;
        int g = 0;
        uint32_t parity = 0;
        const double2* stage_k = reinterpret_cast<const double2*>(stages + k * kWs4StageDoubles) + lane;
        for (int t = k; t < H; t += C) {
            State x;
            x.v = vn;
            x.w = wn;
            ti += tstride;
            if (on && t + C < H) {
                vn = V3{__ldg(a.tw[0] + ti), __ldg(a.tw[1] + ti), __ldg(a.tw[2] + ti)};
                wn = V3{__ldg(a.tw[3] + ti), __ldg(a.tw[4] + ti), __ldg(a.tw[5] + ti)};
            }
            ptx::mbar_wait(full0 + 8 * g, parity);
            const double2* in = stage_k + g * (C * kWs4StageDoubles / 2);
            const double2 a0 = in[0 * kWarp], a1 = in[1 * kWarp], a2 = in[2 * kWarp], a3 = in[3 * kWarp],
                          a4 = in[4 * kWarp], a5 = in[5 * kWarp], a7 = in[7 * kWarp];
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(empty0 + 8 * g);   // one of the C arrivals that free the group
            x.p = V3{a0.x, a0.y, a1.x};
            x.e1 = V3{a2.x, a2.y, a3.x};
            x.e2 = V3{a4.x, a4.y, a5.x};
            x.R02 = 0.0; x.R12 = 0.0;
            x.R22 = a7.x;
            x.p0 = p0; x.n1 = n1; x.n2 = n2;
            Result r;
            eval_contact<M_WRENCH>(x, q, r);
            if (on) {
                const V3 df = r.force - V3{a.ref[0], a.ref[1], a.ref[2]};
                const V3 dt = r.torque - V3{a.ref[3], a.ref[4], a.ref[5]};
                acc = acc + (a.wf * (df.x * df.x + df.y * df.y + df.z * df.z) +
                             a.wt * (dt.x * dt.x + dt.y * dt.y + dt.z * dt.z));
            }
            if (++g == NG) {
                g = 0;
                parity ^= 1u;
            }
        }
        cst[lane * C + k] = acc;    // chains past the end: 0, never read
    }

    // ---------------- fused reduction (as in the third form) ----------------------------------------
    __syncthreads();
    if (warp != 0) return;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    CostIdx mine{inf, 0x7fffffffffffffffLL};
    {
        const int feet = a.feet;
        const long long ro = wbase / feet + lane;          // 32 % feet == 0: tiles hold whole rollouts
        if (lane < kWarp / feet && ro < a.n_rollouts) {
            const double* p = cst + lane * feet * C;
            double sum = 0.0;
            for (int j = 0; j < feet * C; ++j) sum += p[j];
            if (a.cost) a.cost[ro] = sum;
            mine.cost = sum;
            mine.idx = a.index_base + ro;
            if (!(sum == sum)) mine = CostIdx{inf, 0x7fffffffffffffffLL};   // NaN never wins
        }
    }
    mine = warp_best(mine);
    if (lane == 0) {
        a.block_best[blockIdx.x] = mine;
        __threadfence();
        const unsigned int done = atomicAdd(a.counter, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncwarp();
    if (!s_last) return;
    __threadfence();
    CostIdx bb{inf, 0x7fffffffffffffffLL};
    for (unsigned int j = lane; j < gridDim.x; j += kWarp) {
        CostIdx cand;
        cand.cost = *reinterpret_cast<volatile double*>(&a.block_best[j].cost);
        cand.idx = *reinterpret_cast<volatile long long*>(&a.block_best[j].idx);
        if (better(cand.cost, cand.idx, bb.cost, bb.idx)) bb = cand;
    }
    bb = warp_best(bb);
    if (bb.idx == 0x7fffffffffffffffLL) bb.idx = -1;  // nothing comparable (empty / all NaN)
    if (lane == 0) {
        *a.best = bb;
        *a.counter = 0u;
    }
    if (a.p2p.nranks > 0) {   // fused collective: this rank's pair goes straight to the peers' mailboxes
        const CostIdx gbest = p2p_exchange_warp(a.p2p, bb, lane);
        if (lane == 0) *a.p2p.out = gbest;
    }
}

// ------------------------------------------------------------------------------------------------
// Fifth form: the hand-over unit is a BOX of eight steps, the producer's step loop is straight-line
// code, and nothing but the pose recurrence is left on the producer warp.
//
// ncu on the third form (profiles/r02_ncu_rollout_ws3_details.txt): the lone producer warp issues
// one instruction every 3.2 cycles -- 124 instructions and 391 cycles per step with the Baumgarte
// term.  The recurrence alone, timed in isolation (tools/micro/kin_step_lat.cu), takes 191 cycles
// per step (75 FP64 instructions at 2.3 issue cycles each, chain k -> det -> 1/det -> beta -> FMA
// ~105 cycles): half of the producer's time was control -- per step five branches, seven integer
// compares, fourteen register moves rotating the prefetched twist, a try_wait and an arrive every
// third step; per box an elected lane issuing six TMA copies while 31 lanes wait.  A single warp
// has nothing else to issue while a branch resolves or an mbarrier answers (~90 cycles).  Here
//   * a pose stage group IS a twist box: eight steps.  The producer waits and signals once per box;
//     the eight steps in between are one basic block with immediate shared-memory offsets; only the
//     last, partial box runs a rolled loop;
//   * the barriers of box b + 1 are TESTED (mbarrier.test_wait, non-blocking) in the middle of box
//     b, so their latency overlaps the arithmetic and the box border costs no wait in the steady
//     state; a blocking wait runs only when a test said "not yet";
//   * a LOADER warp (one lane) owns the TMA descriptors: it waits for the consumers to release a
//     twist slot and issues the six tensor copies, up to four boxes ahead of the producer;
//   * consumers read the twists of their steps from the SAME box in shared memory (six LDS) instead
//     of global memory (the third form spends ~45 integer instructions per step on six 64-bit
//     plane pointers); every consumer owns a fixed range of the eight steps of a box (the last box
//     of the horizon is dealt round the consumers step by step: nothing follows to hide a long tail);
//   * warp roles follow the scheduler map measured in tools/micro/fp64_lat.cu and warp_slots.cu
//     (see Ws5Cfg): the producer shares its FP64 pipe with the idle loader and, when two CTAs share
//     an SM, with the lightest consumer of the other tile;
//   * two rings: four twist boxes (released by the consumers) and three pose groups.
//   * programmatic dependent launch in its LATE form (signal after the step loops, wait before the
//     first global access), so the next launch's latency and prologue overlap this one's tail.
// Reduction, arg-min and peer exchange are fused as in the third form.  Same preconditions.
// Measured (profiles/r02_rollout_*.log): 30.8 -> 21.1 us per 4096 x 2 x 100 step with rho = 0.01.
// ------------------------------------------------------------------------------------------------

constexpr int kWs5TwSlots = 4;
constexpr int kWs5PoseSlots = 3;
constexpr int kWs5PoseBytes = kWs3BoxSteps * kWs2StageDoubles * 8;   // 20 480: eight stages of (p, e1, e2, R22) x 32 lanes

// Warp roles.  Warp w of a CTA runs on sub-partition (w + r) mod 4, and when two CTAs share an SM the
// second one's r is the first one's + 1 (tools/micro/warp_slots.cu: warp ids 0 1 2 3 4 5 6 7 and
// 9 10 11 8 13 14 15 12), so warp i of one CTA shares a scheduler with warp i + 1 of the other:
// warps 1 and 3 sit beside the OTHER tile's producer.  Layouts (steps of every eight-step box):
//   0: five warps;  producer 0, loader 4, consumers 1 2 3 take steps 0-2 3-5 6-7
//   1: eight warps; producer 0, loader 4, consumers 2 6 1 3 take steps 0-2 3-5 6 7 (the two warps
//      that share a scheduler with a producer get one step each), warps 5 7 idle
//   2: eight warps; consumers 2 6 1 3 take two steps each
struct Ws5Role {
    int k;       // consumer index (column of the partial-cost table), -1: none
    int first;   // first step of the box
    int count;
};

template <int LAYOUT>
struct Ws5Cfg {
    static constexpr int kConsumers = LAYOUT == 0 ? 3 : 4;
    static constexpr int kWarps = LAYOUT == 0 ? 5 : 8;
    static constexpr int kThreads = kWarp * kWarps;
    static constexpr int kBarBytes = 128;
    static constexpr int kSmemBytes = kWs5TwSlots * kWs3BoxBytes + kWs5PoseSlots * kWs5PoseBytes + kBarBytes +
                                      kWarp * kConsumers * 8;
    __device__ static Ws5Role role(int warp)
    {
        if (LAYOUT == 0) {
            if (warp >= 1 && warp <= 3) return Ws5Role{warp - 1, 3 * (warp - 1), warp == 3 ? 2 : 3};
            return Ws5Role{-1, 0, 0};
        }
        const bool weighted = LAYOUT == 1;
        switch (warp) {
        case 2: return weighted ? Ws5Role{0, 0, 3} : Ws5Role{0, 0, 2};
        case 6: return weighted ? Ws5Role{1, 3, 3} : Ws5Role{1, 2, 2};
        case 1: return weighted ? Ws5Role{2, 6, 1} : Ws5Role{2, 4, 2};
        case 3: return weighted ? Ws5Role{3, 7, 1} : Ws5Role{3, 6, 2};
        default: return Ws5Role{-1, 0, 0};
        }
    }
};

// Rollout costs of one 32-chain tile from the consumers' partial sums (cst[lane][parts], summed in
// index order like ccm_cost_reduce_kernel), arg-min over the tile, and -- in the last CTA to get
// here -- over the grid, plus the fused peer exchange.  Called by warp 0 after a __syncthreads().
__device__ __forceinline__ void rollout_tile_reduce(const RolloutArgs& a, const double* cst, int parts,
                                                    long long wbase, int lane, bool* s_last)
{
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    CostIdx mine{inf, 0x7fffffffffffffffLL};
    {
        const int feet = a.feet;
        const long long ro = wbase / feet + lane;          // 32 % feet == 0: tiles hold whole rollouts
        if (lane < kWarp / feet && ro < a.n_rollouts) {
            const double* p = cst + lane * feet * parts;
            double sum = 0.0;
            for (int j = 0; j < feet * parts; ++j) sum += p[j];
            if (a.cost) a.cost[ro] = sum;
            mine.cost = sum;
            mine.idx = a.index_base + ro;
            if (!(sum == sum)) mine = CostIdx{inf, 0x7fffffffffffffffLL};   // NaN never wins
        }
    }
    mine = warp_best(mine);
    if (lane == 0) {
        a.block_best[blockIdx.x] = mine;
        __threadfence();
        const unsigned int done = atomicAdd(a.counter, 1u);
        *s_last = (done == gridDim.x - 1);
    }
    __syncwarp();
    if (!*s_last) return;
    __threadfence();
    CostIdx b{inf, 0x7fffffffffffffffLL};
    for (unsigned int j = lane; j < gridDim.x; j += kWarp) {
        CostIdx cand;
        cand.cost = *reinterpret_cast<volatile double*>(&a.block_best[j].cost);
        cand.idx = *reinterpret_cast<volatile long long*>(&a.block_best[j].idx);
        if (better(cand.cost, cand.idx, b.cost, b.idx)) b = cand;
    }
    b = warp_best(b);
    if (b.idx == 0x7fffffffffffffffLL) b.idx = -1;  // nothing comparable (empty / all NaN)
    if (lane == 0) {
        *a.best = b;
        *a.counter = 0u;
    }
    if (a.p2p.nranks > 0) {   // fused collective: this rank's pair goes straight to the peers' mailboxes
        const CostIdx gbest = p2p_exchange_warp(a.p2p, b, lane);
        if (lane == 0) *a.p2p.out = gbest;
    }
}

template <bool HET, bool BAUM, int LAYOUT>
__global__ void __launch_bounds__(Ws5Cfg<LAYOUT>::kThreads)
ccm_rollout_ws5_kernel(const __grid_constant__ RolloutArgs a)
{
    using Cfg = Ws5Cfg<LAYOUT>;
    constexpr int C = Cfg::kConsumers;
    constexpr int BS = kWs3BoxSteps;
    constexpr int NT = kWs5TwSlots, NP = kWs5PoseSlots;
    constexpr int PL = BS * kWarp;                       // doubles per twist plane of a box
    constexpr int kLoaderWarp = 4;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long wbase = static_cast<long long>(blockIdx.x) * kWarp;
    const long long c = wbase + lane;
    const bool on = c < a.chains;
    const int H = a.horizon;
    const int nbox = (H + BS - 1) / BS;

    double* twbuf = reinterpret_cast<double*>(smem_raw);                       // [NT][plane][step][lane]
    double* poses = twbuf + NT * kWs3BoxBytes / 8;                             // [NP][step][5 double2][lane]
    const uint32_t bars = ptx::smem_addr(poses + NP * kWs5PoseBytes / 8);
    const uint32_t twfull0 = bars;                    // NT barriers: a twist box has landed (TMA bytes)
    const uint32_t twempty0 = twfull0 + 8 * NT;       // NT barriers, C arrivals: the consumers have read it
    const uint32_t full0 = twempty0 + 8 * NT;         // NP barriers, 1 arrival: a pose group is written
    const uint32_t empty0 = full0 + 8 * NP;           // NP barriers, C arrivals: a pose group is consumed
    double* cst = poses + NP * kWs5PoseBytes / 8 + Cfg::kBarBytes / 8;         // [32][C] partial costs
    if (threadIdx.x == 0) {
        for (int i = 0; i < NT; ++i) {
            ptx::mbar_init(twfull0 + 8 * i, 1);
            ptx::mbar_init(twempty0 + 8 * i, C);
        }
        for (int i = 0; i < NP; ++i) {
            ptx::mbar_init(full0 + 8 * i, 1);
            ptx::mbar_init(empty0 + 8 * i, C);
        }
        ptx::fence_mbar_init();
    }
    if (warp == kLoaderWarp && lane < 6) ptx::prefetch_tensormap(&a.twmap[lane]);   // parameters: safe before the wait
    // Programmatic dependent launch, LATE form: this grid's CTAs may become resident while the
    // previous kernel of the stream drains (its CTAs signal after their step loops, below), but
    // nothing global is touched before that kernel has completed.  Signalling at the START (as the
    // streaming kernels do) parks the next launch's CTAs beside a latency-bound kernel and slows it.
    ptx::grid_dep_wait();
    __syncthreads();

    if (warp == kLoaderWarp) {
        // ---------------- loader: twist boxes by TMA, as far ahead as the ring allows -------------
        if (lane == 0) {
            for (int b = 0; b < nbox; ++b) {
                const int slot = b & (NT - 1);
                if (b >= NT) {   // the slot held box b - NT: every consumer must have read it
                    ptx::mbar_wait(twempty0 + 8 * slot, ((b - NT) / NT) & 1);
                    ptx::fence_async_smem();
                }
                const uint32_t bar = twfull0 + 8 * slot;
                const uint32_t dst = ptx::smem_addr(twbuf) + slot * kWs3BoxBytes;
                ptx::mbar_arrive_expect_tx(bar, kWs3BoxBytes);
#pragma unroll
                for (int j = 0; j < 6; ++j)
                    ptx::tma_load_2d(dst + j * (PL * 8), &a.twmap[j], static_cast<int>(wbase), b * BS, bar);
            }
        }
    } else if (warp == 0) {
        // ---------------- producer: the pose recurrence, one basic block per box ------------------
        Pose s{};
        if (on) {
            s.p = V3{__ldg(a.pos0[0] + c), __ldg(a.pos0[1] + c), __ldg(a.pos0[2] + c)};
            s.c0 = V3{__ldg(a.rot0[0] + c), __ldg(a.rot0[3] + c), __ldg(a.rot0[6] + c)};
            s.c1 = V3{__ldg(a.rot0[1] + c), __ldg(a.rot0[4] + c), __ldg(a.rot0[7] + c)};
            s.c2 = V3{__ldg(a.rot0[2] + c), __ldg(a.rot0[5] + c), __ldg(a.rot0[8] + c)};
        }
        const double half_rho = a.half_rho, dT = a.dT;
        auto step = [&](const double* tw, double2* o, int q) {   // publish the pose of step q, then integrate it
            const double* r = tw + q * kWarp;
            const V3 v{r[0], r[PL], r[2 * PL]};
            const V3 w{r[3 * PL], r[4 * PL], r[5 * PL]};
            double2* oq = o + q * (5 * kWarp);
            oq[0 * kWarp] = make_double2(s.p.x, s.p.y);
            oq[1 * kWarp] = make_double2(s.p.z, s.c0.x);
            oq[2 * kWarp] = make_double2(s.c0.y, s.c0.z);
            oq[3 * kWarp] = make_double2(s.c1.x, s.c1.y);
            oq[4 * kWarp] = make_double2(s.c1.z, s.c2.z);
            kin_euler_step<BAUM>(s, v, w, half_rho, dT);
        };
        int ps = 0;                        // pose slot of box b (b mod NP)
        uint32_t pose_use = 0;             // b div NP
        bool tw_ready = false, pose_free = true;   // what the tests issued during the previous box found
        for (int b = 0; b < nbox; ++b) {
            const int ts = b & (NT - 1);
            if (!tw_ready) ptx::mbar_wait(twfull0 + 8 * ts, (b / NT) & 1);
            if (!pose_free) ptx::mbar_wait(empty0 + 8 * ps, (pose_use - 1) & 1);   // pose group of box b - NP consumed
            const double* tw = twbuf + ts * (kWs3BoxBytes / 8) + lane;
            double2* o = reinterpret_cast<double2*>(poses + ps * (kWs5PoseBytes / 8)) + lane;
            // the next box's barriers, tested while this box is integrated
            const int nps = ps + 1 == NP ? 0 : ps + 1;
            const uint32_t nuse = ps + 1 == NP ? pose_use + 1 : pose_use;
            auto test_next = [&]() {
                tw_ready = ptx::mbar_test(twfull0 + 8 * ((b + 1) & (NT - 1)), ((b + 1) / NT) & 1);
                pose_free = (b + 1 < NP) || ptx::mbar_test(empty0 + 8 * nps, (nuse - 1) & 1);
            };
            if ((b + 1) * BS <= H) {
#pragma unroll
                for (int q = 0; q < BS; ++q) {
                    if (q == BS - 3) test_next();
                    step(tw, o, q);
                }
            } else {
#pragma unroll 1
                for (int q = 0; q < H - b * BS; ++q) step(tw, o, q);
            }
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(full0 + 8 * ps);
            ps = nps;
            pose_use = nuse;
        }
        if (on && a.write_final) {
            a.pos_out[0][c] = s.p.x; a.pos_out[1][c] = s.p.y; a.pos_out[2][c] = s.p.z;
            a.rot_out[0][c] = s.c0.x; a.rot_out[1][c] = s.c1.x; a.rot_out[2][c] = s.c2.x;
            a.rot_out[3][c] = s.c0.y; a.rot_out[4][c] = s.c1.y; a.rot_out[5][c] = s.c2.y;
            a.rot_out[6][c] = s.c0.z; a.rot_out[7][c] = s.c1.z; a.rot_out[8][c] = s.c2.z;
        }
    } else if (Cfg::role(warp).k >= 0) {
        // ---------------- consumer: contact wrench + cost of its steps of every box ---------------
        const Ws5Role role = Cfg::role(warp);
        const int k = role.k;
        V3 p0{}, n1{}, n2{};
        Prm q = a.uni;
        if (on) {
            p0 = V3{__ldg(a.nul[0] + c), __ldg(a.nul[1] + c), __ldg(a.nul[2] + c)};
            n1 = V3{__ldg(a.nul[3] + c), __ldg(a.nul[6] + c), __ldg(a.nul[9] + c)};
            n2 = V3{__ldg(a.nul[4] + c), __ldg(a.nul[7] + c), __ldg(a.nul[10] + c)};
            if constexpr (HET)
                q = make_prm(__ldg(a.prm[0] + c), __ldg(a.prm[1] + c), __ldg(a.prm[2] + c),
                             __ldg(a.prm[3] + c));
        }
        const V3 fref{a.ref[0], a.ref[1], a.ref[2]}, tref{a.ref[3], a.ref[4], a.ref[5]};
        const double wf = a.wf, wt = a.wt;
        double acc = 0.0;
        int ps = 0;
        uint32_t pose_use = 0;
        for (int b = 0; b < nbox; ++b) {
            const int ts = b & (NT - 1);
            ptx::mbar_wait(full0 + 8 * ps, pose_use & 1);
            ptx::mbar_wait(twfull0 + 8 * ts, (b / NT) & 1);   // landed long ago; makes the TMA's writes visible to this warp
            const double* tw = twbuf + ts * (kWs3BoxBytes / 8) + lane;
            const double2* in = reinterpret_cast<const double2*>(poses + ps * (kWs5PoseBytes / 8)) + lane;
            const int steps = min(BS, H - b * BS);
            // The last box has nothing behind it to hide an uneven split: its steps go round the
            // consumers one by one, so the tail after the producer's last step is ceil(steps / C)
            // evaluations long instead of role.count.
            const bool tail = b == nbox - 1;
            const int first = tail ? k : role.first;
            const int last = tail ? steps : min(role.first + role.count, steps);
            const int stride = tail ? C : 1;
#pragma unroll 1
            for (int s = first; s < last; s += stride) {
                {
                    const double* r = tw + s * kWarp;
                    const double2* is = in + s * (5 * kWarp);
                    const double2 a0 = is[0 * kWarp], a1 = is[1 * kWarp], a2 = is[2 * kWarp], a3 = is[3 * kWarp],
                                  a4 = is[4 * kWarp];
                    State x;
                    x.v = V3{r[0], r[PL], r[2 * PL]};
                    x.w = V3{r[3 * PL], r[4 * PL], r[5 * PL]};
                    x.p = V3{a0.x, a0.y, a1.x};
                    x.e1 = V3{a1.y, a2.x, a2.y};
                    x.e2 = V3{a3.x, a3.y, a4.x};
                    x.R02 = 0.0; x.R12 = 0.0;
                    x.R22 = a4.y;
                    x.p0 = p0; x.n1 = n1; x.n2 = n2;
                    Result res;
                    eval_contact<M_WRENCH>(x, q, res);
                    if (on) {
                        const V3 df = res.force - fref;
                        const V3 dt = res.torque - tref;
                        acc = acc + (wf * (df.x * df.x + df.y * df.y + df.z * df.z) +
                                     wt * (dt.x * dt.x + dt.y * dt.y + dt.z * dt.z));
                    }
                }
            }
            __syncwarp();
            if (lane == 0) {   // this warp's share of the C arrivals that free the box and the group
                ptx::mbar_arrive(empty0 + 8 * ps);
                ptx::mbar_arrive(twempty0 + 8 * ts);
            }
            if (++ps == NP) {
                ps = 0;
                ++pose_use;
            }
        }
        cst[lane * C + k] = acc;    // chains past the end: 0, never read
    }

    ptx::grid_dep_launch_dependents();   // the next launch may take the slots this CTA is about to free
    __syncthreads();
    if (warp == 0) rollout_tile_reduce(a, cst, C, wbase, lane, &s_last);
}

// ------------------------------------------------------------------------------------------------
// J^T * wrench accumulation
// ------------------------------------------------------------------------------------------------

constexpr int kGfStages = 4;    // Jacobian blocks in flight per warp
constexpr int kGfMaxChunks = 4; // ncols <= 128

struct GenForceArgs {
    const double* in[30];
    const double* prm[4];
    Prm uni;
    const double* jac;     // [n_contacts][6][ncols] row-major
    const double* base;    // [n_systems][ncols] or nullptr
    double* out;           // [n_systems][ncols]
    double* wrench[6];     // optional planes (all nullptr when not wanted)
    long long n_systems;
    int cps;               // contacts per system (1..32)
    int ncols;
    int sys_per_warp;      // 32 / cps
    int jac_bulk;          // jac 16-byte aligned -> TMA ring; else direct loads
    int want_wrench;
    int cps_stage;         // consecutive contacts per ring stage (about 2 KB of Jacobians)
    int stage_bytes;       // per-stage shared-memory bytes (cps_stage*48*ncols rounded up to 128)
    int row_bytes;         // > 0: per-warp shared-memory bytes for the warp's base / out rows
    int base_negate;       // != 0: start from -base (the reference starts from the negated bias forces,
                           // FloatingBaseSystemDynamics.cpp:191-196); the sign flip is exact
};

// NCH = ceil(ncols / 32): column chunks a lane owns (compile-time so dead chunks cost nothing);
// BULK: Jacobians through the TMA ring (16-byte aligned) or direct loads.
//
// The kernel is ISSUE-bound before it is HBM-bound if the per-contact instruction count is not kept
// down (ncu on the first versions: 74-77 % issue slots busy; ~120-150 warp instructions per contact,
// whatever the Jacobian's width -- so narrow Jacobians got 50 % of HBM).  Hence:
//   * a ring stage holds `cps_stage` CONSECUTIVE contacts (about 2 KB): one mbarrier wait and one
//     re-arm + bulk copy per stage, not per contact;
//   * Jacobian reads are shared-memory loads off one per-lane base address (BULK is compile-time, so
//     no generic addressing); the wrench is three broadcast LDS.128;
//   * stage / system bookkeeping is incremental (no divisions, loop invariants in registers);
//   * the warp's base / out rows are staged through shared memory with one bulk copy each (read per
//     system they cost a global-load latency each).
template <bool HET, int NCH, bool BULK>
__global__ void __launch_bounds__(128)
ccm_genforce_kernel(const __grid_constant__ GenForceArgs a)
{
    constexpr unsigned LIVE = live_planes(M_WRENCH);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long wid = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp;
    const long long sys0 = wid * a.sys_per_warp;
    if (sys0 >= a.n_systems) return;  // warp-uniform
    const int nsys = static_cast<int>(min64(a.sys_per_warp, a.n_systems - sys0));
    const int cps = a.cps, ncols = a.ncols, cpst = a.cps_stage, stage_bytes = a.stage_bytes;
    const int ncont = nsys * cps;
    const long long c0 = sys0 * cps;           // first contact of this warp
    const int jd = 6 * ncols;                  // doubles of one contact's Jacobian
    const int nstage = (ncont + cpst - 1) / cpst;

    // per warp: kGfStages Jacobian stages | 32 wrenches (32 x 48 B) | kGfStages + 1 mbarriers |
    //           the warp's base / out rows
    const int per_warp = kGfStages * stage_bytes + kWarp * 48 + 128 + a.row_bytes;
    unsigned char* ws = smem_raw + static_cast<size_t>(warp) * per_warp;
    double* wsm = reinterpret_cast<double*>(ws + kGfStages * stage_bytes);
    const uint32_t bar0 = ptx::smem_addr(ws + kGfStages * stage_bytes + kWarp * 48);
    const uint32_t rbar = bar0 + 8 * kGfStages;
    double* rows = reinterpret_cast<double*>(ws + kGfStages * stage_bytes + kWarp * 48 + 128);
    const uint32_t stage0 = ptx::smem_addr(ws);
    const double* jac0 = a.jac + c0 * jd;
    const long long row0 = sys0 * ncols;
    const uint32_t rbytes = static_cast<uint32_t>(nsys) * ncols * 8u;
    const bool staged = a.row_bytes > 0 && ((row0 | (static_cast<long long>(nsys) * ncols)) & 1) == 0;

    auto arm = [&](int q) {   // lane 0: bulk copy of stage q (contacts q*cpst ..) into its ring slot
        const int first = q * cpst;
        const uint32_t bytes = static_cast<uint32_t>(min(cpst, ncont - first)) * jd * 8u;
        const uint32_t bar = bar0 + 8 * (q & (kGfStages - 1));
        ptx::mbar_arrive_expect_tx(bar, bytes);
        ptx::bulk_g2s(stage0 + (q & (kGfStages - 1)) * stage_bytes, jac0 + static_cast<long long>(first) * jd,
                      bytes, bar);
    };

    ptx::grid_dep_launch_dependents();   // PDL: see ccm_soa_kernel
    if (lane == 0 && (BULK || staged)) {
#pragma unroll
        for (int s = 0; s <= kGfStages; ++s) ptx::mbar_init(bar0 + 8 * s, 1);
        ptx::fence_mbar_init();
    }
    ptx::grid_dep_wait();
    if (lane == 0) {
        if (staged && a.base) {
            ptx::mbar_arrive_expect_tx(rbar, rbytes);
            ptx::bulk_g2s(ptx::smem_addr(rows), a.base + row0, rbytes, rbar);
        }
        if constexpr (BULK) {
#pragma unroll
            for (int q = 0; q < kGfStages; ++q)
                if (q < nstage) arm(q);
        }
    }
    __syncwarp();

    // ---- wrench of this lane's contact --------------------------------------------------------
    const bool on = lane < ncont;
    const long long i = c0 + lane;
    double x[30] = {};
    load_live_planes<LIVE>(a.in, i, on, x);
    const Prm q = load_params<HET>(a.prm, a.uni, i, on);
    Result r;
    eval_contact<M_WRENCH>(state_from_planes(x), q, r);
    if (a.want_wrench && on) store_wrench(a.wrench, i, r);
    {
        double2* o = reinterpret_cast<double2*>(wsm) + lane * 3;
        o[0] = make_double2(r.force.x, r.force.y);
        o[1] = make_double2(r.force.z, r.torque.x);
        o[2] = make_double2(r.torque.y, r.torque.z);
    }
    __syncwarp();

    // ---- lanes own columns; stages, and the contacts inside a stage, are visited in order ------
    bool mine[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) mine[ch] = ch * kWarp + lane < ncols;
    if (staged && a.base) ptx::mbar_wait(rbar, 0);
    int sys = 0, cin = 0;            // system / contact-in-system of the contact being added
    double acc[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) acc[ch] = 0.0;
    const double2* wv = reinterpret_cast<const double2*>(wsm);
    int slot = 0;
    uint32_t parity = 0;
    for (int sq = 0; sq < nstage; ++sq) {
        const int first = sq * cpst;
        const int cnt = min(cpst, ncont - first);
        const double* J;
        if constexpr (BULK) {
            ptx::mbar_wait(bar0 + 8 * slot, parity);
            J = reinterpret_cast<const double*>(ws + slot * stage_bytes) + lane;
        } else {
            J = jac0 + static_cast<long long>(first) * jd + lane;
        }
        for (int j = 0; j < cnt; ++j, J += jd, wv += 3) {
            if (cin == 0) {   // a new system starts: acc = base row
                const long long row = (sys0 + sys) * ncols + lane;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (staged) acc[ch] = (mine[ch] && a.base) ? rows[sys * ncols + lane + ch * kWarp] : 0.0;
                    else acc[ch] = (mine[ch] && a.base) ? __ldcs(a.base + row + ch * kWarp) : 0.0;
                    if (a.base_negate) acc[ch] = -acc[ch];
                }
            }
            const double2 w01 = wv[0], w23 = wv[1], w45 = wv[2];
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                if (mine[ch]) {
                    // (J^T w)[col], rows in order; then known += product  (:224-225)
                    const double* Jc = J + ch * kWarp;
                    double t;
                    if constexpr (BULK) {
                        t = Jc[0] * w01.x;
                        t += Jc[ncols] * w01.y;
                        t += Jc[2 * ncols] * w23.x;
                        t += Jc[3 * ncols] * w23.y;
                        t += Jc[4 * ncols] * w45.x;
                        t += Jc[5 * ncols] * w45.y;
                    } else {
                        t = __ldcs(Jc) * w01.x;
                        t += __ldcs(Jc + ncols) * w01.y;
                        t += __ldcs(Jc + 2 * ncols) * w23.x;
                        t += __ldcs(Jc + 3 * ncols) * w23.y;
                        t += __ldcs(Jc + 4 * ncols) * w45.x;
                        t += __ldcs(Jc + 5 * ncols) * w45.y;
                    }
                    acc[ch] = acc[ch] + t;
                }
            }
            if (++cin == cps) {   // the system is complete: its row leaves
                const long long row = (sys0 + sys) * ncols + lane;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (!mine[ch]) continue;
                    if (staged) rows[sys * ncols + lane + ch * kWarp] = acc[ch];
                    else __stcs(a.out + row + ch * kWarp, acc[ch]);
                }
                cin = 0;
                ++sys;
            }
        }
        if constexpr (BULK) {
            __syncwarp();   // every lane is done with this stage
            if (lane == 0 && sq + kGfStages < nstage) arm(sq + kGfStages);
            if (++slot == kGfStages) {
                slot = 0;
                parity ^= 1u;
            }
        }
    }
    if (staged) {   // the warp's rows leave with one bulk store
        ptx::fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            ptx::bulk_s2g(a.out + row0, ptx::smem_addr(rows), rbytes);
            ptx::bulk_commit();
            ptx::bulk_wait_read_all();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Narrow Jacobians (ncols <= 16): lane-packed form.
//
// With lanes owning columns, a 6-column Jacobian keeps 6 of 32 lanes busy and the kernel above is
// issue-bound at ~60 % of HBM (12 columns: ~80 %).  Here the warp is cut into G = 32 / NCP lane
// groups (NCP = 4, 8 or 16 >= ncols) and every group owns a whole SYSTEM: lane (g, col) accumulates
// column col of system it*G + g over that system's contacts, in order -- the same products and the
// same order of additions as the kernel above (and the reference's loop,
// FloatingBaseSystemDynamics.cpp:199-226), so the results are bit-identical; no shuffles are needed
// because no sum crosses a group.  A ring stage holds the Jacobians of G consecutive systems
// (G * cps contacts, contiguous in memory): one mbarrier wait + one re-arm per G systems.  The
// instruction stream per iteration is the one of the kernel above, but it now covers G contacts.
// NST = ring stages per warp: 2 by default (twice the warps per SM of a four-stage ring, measured
// 84 -> 107 % of HBM at 6 columns), 4 with BLF_CCM_TUNE_GF_STAGES=4.
// (A first lane-packed attempt in round 1 split the CONTACTS of one system over the groups and
// needed ordered shuffles; it gained nothing and was removed.)
// ------------------------------------------------------------------------------------------------
template <bool HET, int NCP, int NST>
__global__ void __launch_bounds__(128)
ccm_genforce_packed_kernel(const __grid_constant__ GenForceArgs a)
{
    constexpr unsigned LIVE = live_planes(M_WRENCH);
    constexpr int G = kWarp / NCP;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long wid = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp;
    const long long sys0 = wid * a.sys_per_warp;
    if (sys0 >= a.n_systems) return;  // warp-uniform
    const int nsys = static_cast<int>(min64(a.sys_per_warp, a.n_systems - sys0));
    const int cps = a.cps, ncols = a.ncols, stage_bytes = a.stage_bytes;
    const int ncont = nsys * cps;
    const long long c0 = sys0 * cps;
    const int jd = 6 * ncols;
    const int nstage = (nsys + G - 1) / G;     // G systems per stage

    const int per_warp = NST * stage_bytes + kWarp * 48 + 128 + a.row_bytes;
    unsigned char* ws = smem_raw + static_cast<size_t>(warp) * per_warp;
    double* wsm = reinterpret_cast<double*>(ws + NST * stage_bytes);
    const uint32_t bar0 = ptx::smem_addr(ws + NST * stage_bytes + kWarp * 48);
    const uint32_t rbar = bar0 + 8 * NST;
    double* rows = reinterpret_cast<double*>(ws + NST * stage_bytes + kWarp * 48 + 128);
    const uint32_t stage0 = ptx::smem_addr(ws);
    const double* jac0 = a.jac + c0 * jd;
    const long long row0 = sys0 * ncols;
    const uint32_t rbytes = static_cast<uint32_t>(nsys) * ncols * 8u;
    const bool staged = a.row_bytes > 0 && ((row0 | (static_cast<long long>(nsys) * ncols)) & 1) == 0;

    auto arm = [&](int q) {   // lane 0: the Jacobians of systems q*G .. q*G+G-1 into ring slot q % NST
        const int first = q * G * cps;
        const uint32_t bytes = static_cast<uint32_t>(min(G * cps, ncont - first)) * jd * 8u;
        const uint32_t bar = bar0 + 8 * (q & (NST - 1));
        ptx::mbar_arrive_expect_tx(bar, bytes);
        ptx::bulk_g2s(stage0 + (q & (NST - 1)) * stage_bytes, jac0 + static_cast<long long>(first) * jd,
                      bytes, bar);
    };

    ptx::grid_dep_launch_dependents();   // PDL: see ccm_soa_kernel
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s <= NST; ++s) ptx::mbar_init(bar0 + 8 * s, 1);
        ptx::fence_mbar_init();
    }
    ptx::grid_dep_wait();
    if (lane == 0) {
        if (staged && a.base) {
            ptx::mbar_arrive_expect_tx(rbar, rbytes);
            ptx::bulk_g2s(ptx::smem_addr(rows), a.base + row0, rbytes, rbar);
        }
#pragma unroll
        for (int q = 0; q < NST; ++q)
            if (q < nstage) arm(q);
    }
    __syncwarp();

    // ---- wrench of this lane's contact (as in ccm_genforce_kernel) -----------------------------
    const bool on = lane < ncont;
    const long long i = c0 + lane;
    double x[30] = {};
    load_live_planes<LIVE>(a.in, i, on, x);
    const Prm q = load_params<HET>(a.prm, a.uni, i, on);
    Result r;
    eval_contact<M_WRENCH>(state_from_planes(x), q, r);
    if (a.want_wrench && on) store_wrench(a.wrench, i, r);
    {
        double2* o = reinterpret_cast<double2*>(wsm) + lane * 3;
        o[0] = make_double2(r.force.x, r.force.y);
        o[1] = make_double2(r.force.z, r.torque.x);
        o[2] = make_double2(r.torque.y, r.torque.z);
    }
    __syncwarp();

    // ---- lane (g, col): column col of system it*G + g ------------------------------------------
    const int g = lane / NCP, col = lane % NCP;
    const bool active = col < ncols;
    if (staged && a.base) ptx::mbar_wait(rbar, 0);
    int slot = 0;
    uint32_t parity = 0;
    const int goff = g * cps * jd + (active ? col : 0);      // this group's first Jacobian inside a stage
    for (int sq = 0; sq < nstage; ++sq) {
        const int s = sq * G + g;
        const bool valid = active && s < nsys;
        const int sc = valid ? s : 0;                         // in-bounds addresses for idle lanes
        ptx::mbar_wait(bar0 + 8 * slot, parity);
        const double* J = reinterpret_cast<const double*>(ws + slot * stage_bytes) + (valid ? goff : 0);
        const double2* wv = reinterpret_cast<const double2*>(wsm) + sc * cps * 3;
        const long long row = (sys0 + sc) * ncols + col;
        double acc = 0.0;
        if (valid && a.base) acc = staged ? rows[sc * ncols + col] : __ldcs(a.base + row);
        if (a.base_negate) acc = -acc;
        for (int j = 0; j < cps; ++j, J += jd, wv += 3) {
            const double2 w01 = wv[0], w23 = wv[1], w45 = wv[2];
            // (J^T w)[col], rows in order; then known += product  (:224-225)
            double t = J[0] * w01.x;
            t += J[ncols] * w01.y;
            t += J[2 * ncols] * w23.x;
            t += J[3 * ncols] * w23.y;
            t += J[4 * ncols] * w45.x;
            t += J[5 * ncols] * w45.y;
            acc = acc + t;
        }
        if (valid) {
            if (staged) rows[sc * ncols + col] = acc;
            else __stcs(a.out + row, acc);
        }
        __syncwarp();   // every lane is done with this stage
        if (lane == 0 && sq + NST < nstage) arm(sq + NST);
        if (++slot == NST) {
            slot = 0;
            parity ^= 1u;
        }
    }
    if (staged) {   // the warp's rows leave with one bulk store
        ptx::fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            ptx::bulk_s2g(a.out + row0, ptx::smem_addr(rows), rbytes);
            ptx::bulk_commit();
            ptx::bulk_wait_read_all();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// One ForwardEuler step of System::FloatingBaseDynamicalSystem (ForwardEuler.tpp:19-49: x = x0 + dx * dT
// over the state tuple of FloatingBaseSystemDynamics.h:33-52), every derivative at the state BEFORE the
// step: base position += nu.head<3>() dT, base rotation += (rotation rate of
// FloatingBaseSystemDynamics.cpp:139-145 = the kinematics' formula) dT, joint positions += nu.tail dT,
// nu += acc dT.  Array-of-structures state as the reference holds it (per system: nu[nc], jointPos[nc-6],
// basePos[3], baseRot[9] row-major).
//
// HBM-bound: (5 nc + 12) doubles per system.  A CTA owns a tile of `tile` consecutive systems; in each of
// the five arrays that tile is ONE contiguous run of bytes, so it is brought into shared memory by five 1-D
// bulk copies (TMA engine) signalled on one mbarrier, updated there, and written back by four bulk stores.
// No per-thread global access at all on that path; bytes in flight = tile bytes x resident CTAs.  A tile
// with an odd count (the last one) or arrays that are only 8-byte aligned take the same route with
// per-thread 8-byte async copies (LDGSTS) and plain streaming stores.  The new velocity is built in the
// acceleration's buffer, so nothing reads a value another thread has replaced.  One thread per system
// does the pose (warp 0 mostly; the other warps go on with the elementwise part).
// ------------------------------------------------------------------------------------------------
struct FbdEulerArgs {
    const double* acc;   // [n][nc]
    double* nu;          // [n][nc]   in/out
    double* jp;          // [n][nc-6] in/out (nullptr when nc == 6)
    double* pos;         // [n][3]    in/out
    double* rot;         // [n][9]    in/out, row-major
    double half_rho, dT;
    long long n;
    int nc;
    int tile;            // systems per CTA, even
    int bulk;            // all five arrays 16-byte aligned
    unsigned magic;      // ceil(2^32 / nc): e / nc == __umulhi(e, magic) for e < tile * nc
};

template <bool BAUM>
__global__ void __launch_bounds__(128)
sys_fbd_euler_kernel(const __grid_constant__ FbdEulerArgs a)
{
    extern __shared__ __align__(16) double fbd_sm[];
    __shared__ __align__(8) unsigned long long fbd_bar;
    const int tid = threadIdx.x, nth = blockDim.x;
    const int nc = a.nc, nj = nc - 6, S = a.tile;
    const long long s0 = static_cast<long long>(blockIdx.x) * S;
    const int cnt = static_cast<int>(a.n - s0 < S ? a.n - s0 : S);
    double* s_acc = fbd_sm;              // becomes the new velocity
    double* s_nu = s_acc + S * nc;
    double* s_jp = s_nu + S * nc;
    double* s_pos = s_jp + S * nj;
    double* s_rot = s_pos + S * 3;
    const double* g_acc = a.acc + s0 * nc;
    double* g_nu = a.nu + s0 * nc;
    double* g_jp = a.jp + s0 * nj;
    double* g_pos = a.pos + s0 * 3;
    double* g_rot = a.rot + s0 * 9;
    const bool bulk = a.bulk && !(cnt & 1);   // every run a multiple of 16 bytes
    const int n_nu = cnt * nc, n_jp = cnt * nj;
    if (bulk && tid == 0) {
        ptx::mbar_init(ptx::smem_addr(&fbd_bar), 1);
        ptx::fence_mbar_init();
    }
    ptx::grid_dep_launch_dependents();   // PDL: see ccm_soa_kernel
    ptx::grid_dep_wait();
    if (bulk) {
        __syncthreads();
        const uint32_t bar = ptx::smem_addr(&fbd_bar);
        if (tid == 0) {
            ptx::mbar_arrive_expect_tx(bar, static_cast<uint32_t>((2 * n_nu + n_jp + 12 * cnt) * 8));
            ptx::bulk_g2s(ptx::smem_addr(s_nu), g_nu, n_nu * 8, bar);
            ptx::bulk_g2s(ptx::smem_addr(s_rot), g_rot, cnt * 72, bar);
            ptx::bulk_g2s(ptx::smem_addr(s_pos), g_pos, cnt * 24, bar);
            if (nj > 0) ptx::bulk_g2s(ptx::smem_addr(s_jp), g_jp, n_jp * 8, bar);
            ptx::bulk_g2s(ptx::smem_addr(s_acc), g_acc, n_nu * 8, bar);
        }
        ptx::mbar_wait(bar, 0);
    } else {
        for (int e = tid; e < n_nu; e += nth) {
            ptx::cp_async8(ptx::smem_addr(s_nu + e), g_nu + e);
            ptx::cp_async8(ptx::smem_addr(s_acc + e), g_acc + e);
        }
        for (int e = tid; e < n_jp; e += nth) ptx::cp_async8(ptx::smem_addr(s_jp + e), g_jp + e);
        for (int e = tid; e < cnt * 9; e += nth) ptx::cp_async8(ptx::smem_addr(s_rot + e), g_rot + e);
        for (int e = tid; e < cnt * 3; e += nth) ptx::cp_async8(ptx::smem_addr(s_pos + e), g_pos + e);
        ptx::cp_async_commit();
        ptx::cp_async_wait<0>();
        __syncthreads();
    }
    // pose of system tid (reads the old base twist; nobody writes s_nu)
    for (int s = tid; s < cnt; s += nth) {
        const double* t = s_nu + s * nc;
        double* P = s_pos + 3 * s;
        double* R = s_rot + 9 * s;
        Pose q{V3{P[0], P[1], P[2]}, V3{R[0], R[3], R[6]}, V3{R[1], R[4], R[7]}, V3{R[2], R[5], R[8]}};
        kin_euler_step<BAUM>(q, V3{t[0], t[1], t[2]}, V3{t[3], t[4], t[5]}, a.half_rho, a.dT);
        P[0] = q.p.x; P[1] = q.p.y; P[2] = q.p.z;
        R[0] = q.c0.x; R[1] = q.c1.x; R[2] = q.c2.x;
        R[3] = q.c0.y; R[4] = q.c1.y; R[5] = q.c2.y;
        R[6] = q.c0.z; R[7] = q.c1.z; R[8] = q.c2.z;
    }
    // joint positions += old joint velocity * dT; velocity += acceleration * dT (into the acceleration's buffer)
    for (int e = tid; e < n_nu; e += nth) {
        const int s = static_cast<int>(__umulhi(static_cast<unsigned>(e), a.magic));
        const int q = e - s * nc;
        const double old = s_nu[e];
        if (q >= 6) {
            double* j = s_jp + s * nj + (q - 6);
            *j = fma(old, a.dT, *j);
        }
        s_acc[e] = fma(s_acc[e], a.dT, old);
    }
    if (bulk) {
        ptx::fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            ptx::bulk_s2g(g_nu, ptx::smem_addr(s_acc), n_nu * 8);
            if (nj > 0) ptx::bulk_s2g(g_jp, ptx::smem_addr(s_jp), n_jp * 8);
            ptx::bulk_s2g(g_pos, ptx::smem_addr(s_pos), cnt * 24);
            ptx::bulk_s2g(g_rot, ptx::smem_addr(s_rot), cnt * 72);
            ptx::bulk_commit();
            ptx::bulk_wait_read_all();
        }
    } else {
        __syncthreads();
        for (int e = tid; e < n_nu; e += nth) __stcs(g_nu + e, s_acc[e]);
        for (int e = tid; e < n_jp; e += nth) __stcs(g_jp + e, s_jp[e]);
        for (int e = tid; e < cnt * 9; e += nth) __stcs(g_rot + e, s_rot[e]);
        for (int e = tid; e < cnt * 3; e += nth) __stcs(g_pos + e, s_pos[e]);
    }
}

}  // namespace blfccm
