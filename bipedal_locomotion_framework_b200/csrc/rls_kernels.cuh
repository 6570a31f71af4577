// rls_kernels.cuh -- batched Estimators::RecursiveLeastSquare::advance on sm_100a
// (SURVEY.md section 8(f) row 1; reference: src/Estimators/src/RecursiveLeastSquare.cpp:96-133).
//
// One independent estimator per thread, everything in registers (P <= 4 parameters, M <= 6
// measurements; the contact model has P = 2 [spring, damper], M = 6 [wrench]):
//   K     = P Y^T (lambda R + Y P Y^T)^-1
//   theta = theta + K (z - Y theta)
//   P     = (P - K Y P) / lambda
// Same structure as the reference: the M x M matrix S = lambda R + Y P Y^T is factorised and
// K^T = S^-1 (Y P^T).  S is symmetric positive definite (lambda R > 0 plus a Gram term), so the
// factorisation is an in-register LDL^T on the lower triangle with M reciprocals -- about 350 FP64
// instructions for the contact model, which keeps the kernel HBM-bound (a first version with a full
// Gaussian elimination and 27 true divisions was FP64-bound at 24 % of the HBM roofline).  The
// error is governed by cond(S), as for the reference's LU.  Shortcuts through a P x P system
// (information form, push-through identity) were rejected: their conditioning picks up cond(P),
// which grows by decades when spring and damper variances drift apart (tests caught 2e-12 misses).
// theta and P are updated with the reference's own expressions (including the cancellation-prone
// P - K Y P), so rounding behaves like the reference's.
// HBM: (M*P + M + P + P*P) doubles in, (P + P*P) out per estimator and step; the fused contact
// variant computes Y from the contact state in registers so the regressor never exists in HBM.
#pragma once

#include "ccm_math.cuh"
#include "ccm_ptx.cuh"

namespace blfccm {

// lr[i] = lambda * r[i] (diagonal of lambda R), precomputed on the host: uniform over the batch.
template <int P, int M>
__device__ __forceinline__ void rls_advance(const double (&Y)[M][P], const double (&z)[M],
                                            const double (&lr)[M], double lambda, double (&th)[P],
                                            double (&C)[P][P])
{
    // A = Y C (M x P),  B = Y C^T (M x P)
    double A[M][P], B[M][P];
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
        for (int c = 0; c < P; ++c) {
            double a = 0.0, b = 0.0;
#pragma unroll
            for (int k = 0; k < P; ++k) {
                a += Y[i][k] * C[k][c];
                b += Y[i][k] * C[c][k];
            }
            A[i][c] = a;
            B[i][c] = b;
        }
    // innovation z - Y theta: formed here so that Y and z are dead during the factorisation
    // (register pressure: 172 -> see DESIGN.md section 10)
    double innov[M];
#pragma unroll
    for (int i = 0; i < M; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < P; ++k) acc += Y[i][k] * th[k];
        innov[i] = z[i] - acc;
    }
    // lower triangle of S = lambda R + A Y^T
    double S[M][M];
#pragma unroll
    for (int i = 0; i < M; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double v = (i == j) ? lr[i] : 0.0;
#pragma unroll
            for (int k = 0; k < P; ++k) v += A[i][k] * Y[j][k];
            S[i][j] = v;
        }
    // LDL^T: afterwards S[i][k] (i > k) holds l_ik, inv[k] = 1 / d_k; B is forward-substituted
    double inv[M];
#pragma unroll
    for (int k = 0; k < M; ++k) {
        inv[k] = 1.0 / S[k][k];
        double l[M];                         // l_ik for this column; S[.][k] stays unscaled (l d)
#pragma unroll
        for (int i = k + 1; i < M; ++i) l[i] = S[i][k] * inv[k];
#pragma unroll
        for (int i = k + 1; i < M; ++i) {
#pragma unroll
            for (int j = k + 1; j <= i; ++j) S[i][j] -= l[i] * S[j][k];
#pragma unroll
            for (int c = 0; c < P; ++c) B[i][c] -= l[i] * B[k][c];
        }
#pragma unroll
        for (int i = k + 1; i < M; ++i) S[i][k] = l[i];
    }
#pragma unroll
    for (int kk = 0; kk < M; ++kk) {        // D^-1 then L^T back substitution (counted upwards)
        const int k = M - 1 - kk;
#pragma unroll
        for (int c = 0; c < P; ++c) {
            double acc = B[k][c] * inv[k];
#pragma unroll
            for (int i = k + 1; i < M; ++i) acc -= S[i][k] * B[i][c];
            B[k][c] = acc;                  // B now holds K^T
        }
    }
    // theta += K (z - Y theta)   (innovation formed before the factorisation, see above)
#pragma unroll
    for (int c = 0; c < P; ++c) {
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < M; ++i) acc += B[i][c] * innov[i];
        th[c] += acc;
    }
    // C = (C - K A) / lambda     (the reference's expression)
    double Cn[P][P];
#pragma unroll
    for (int a = 0; a < P; ++a)
#pragma unroll
        for (int c = 0; c < P; ++c) {
            double acc = 0.0;
#pragma unroll
            for (int i = 0; i < M; ++i) acc += B[i][a] * A[i][c];
            Cn[a][c] = (C[a][c] - acc) / lambda;
        }
#pragma unroll
    for (int a = 0; a < P; ++a)
#pragma unroll
        for (int c = 0; c < P; ++c) C[a][c] = Cn[a][c];
}

constexpr int kRlsMaxP = 4, kRlsMaxM = 6;

struct RlsArgs {
    // SoA: plane pointers; AoS: element [0] of each array is the base pointer
    const double* Y[kRlsMaxM * kRlsMaxP];
    const double* z[kRlsMaxM];
    double* theta[kRlsMaxP];
    double* cov[kRlsMaxP * kRlsMaxP];
    double w[kRlsMaxM];        // lambda * r[i]
    double lambda;
    long long n;
};

template <int P, int M, bool AOS>
__global__ void __launch_bounds__(128, (P <= 2 ? 3 : 2))
rls_advance_kernel(const __grid_constant__ RlsArgs a)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    double Y[M][P], z[M], r[M], th[P], C[P][P];
#pragma unroll
    for (int q = 0; q < M; ++q) {
        r[q] = a.w[q];
        z[q] = AOS ? a.z[0][i * M + q] : __ldcs(a.z[q] + i);
#pragma unroll
        for (int c = 0; c < P; ++c)
            Y[q][c] = AOS ? a.Y[0][i * (M * P) + q * P + c] : __ldcs(a.Y[q * P + c] + i);
    }
#pragma unroll
    for (int c = 0; c < P; ++c) {
        th[c] = AOS ? a.theta[0][i * P + c] : __ldcs(a.theta[c] + i);
#pragma unroll
        for (int d = 0; d < P; ++d)
            C[c][d] = AOS ? a.cov[0][i * (P * P) + c * P + d] : __ldcs(a.cov[c * P + d] + i);
    }
    rls_advance<P, M>(Y, z, r, a.lambda, th, C);
#pragma unroll
    for (int c = 0; c < P; ++c) {
        if (AOS) a.theta[0][i * P + c] = th[c];
        else __stcs(a.theta[c] + i, th[c]);
#pragma unroll
        for (int d = 0; d < P; ++d) {
            if (AOS) a.cov[0][i * (P * P) + c * P + d] = C[c][d];
            else __stcs(a.cov[c * P + d] + i, C[c][d]);
        }
    }
}

// Software-pipelined SoA variant.  The plain kernel above is LATENCY-bound at its occupancy (168
// registers -> 12 warps/SM): every warp loads, then computes for ~2 us through six dependent FP64
// reciprocals, and while it computes it has nothing in flight -- 82 % of the HBM peak at 8.4 M
// estimators, 61 % at 819 200 where the first waves also run in lock-step.  Here a block keeps
// walking over tiles of 128 estimators (tile = blockIdx.x + k * gridDim.x) and every thread
// prefetches ITS OWN next estimator with per-thread 8-byte async copies (LDGSTS: no registers held,
// no block-wide synchronisation -- a thread only ever reads what it copied itself, so
// cp.async.wait_group is all the ordering needed) into a two-stage shared-memory ring while it
// computes the current one.  Shared memory: 2 x NIN x 128 x 8 B per block (48 KB for P=2, M=6).
template <int P, int M>
struct RlsPipe {
    static constexpr int NIN = M * P + M + P + P * P;   // planes read per estimator
    static constexpr int STAGES = 2;
    static constexpr int THREADS = 128;
    static constexpr int SMEM_BYTES = STAGES * NIN * THREADS * 8;
};

template <int P, int M, int BLOCKS_PER_SM>
__global__ void __launch_bounds__(128, BLOCKS_PER_SM)
rls_advance_pipe_kernel(const __grid_constant__ RlsArgs a, long long ntiles)
{
    using Cfg = RlsPipe<P, M>;
    constexpr int NIN = Cfg::NIN, T = Cfg::THREADS;
    extern __shared__ __align__(16) double rls_ring[];      // [stage][plane][thread]
    const int tid = threadIdx.x;

    auto issue = [&](int stage, long long tile) {
        const long long i = tile * T + tid;
        if (tile < ntiles && i < a.n) {
            const uint32_t base = ptx::smem_addr(rls_ring + (static_cast<size_t>(stage) * NIN) * T + tid);
            int q = 0;
#pragma unroll
            for (int k = 0; k < M * P; ++k, ++q) ptx::cp_async8(base + q * T * 8, a.Y[k] + i);
#pragma unroll
            for (int k = 0; k < M; ++k, ++q) ptx::cp_async8(base + q * T * 8, a.z[k] + i);
#pragma unroll
            for (int k = 0; k < P; ++k, ++q) ptx::cp_async8(base + q * T * 8, a.theta[k] + i);
#pragma unroll
            for (int k = 0; k < P * P; ++k, ++q) ptx::cp_async8(base + q * T * 8, a.cov[k] + i);
        }
        ptx::cp_async_commit();                             // one group per tile, empty or not
    };

    double r[M];
#pragma unroll
    for (int q = 0; q < M; ++q) r[q] = a.w[q];

    long long tile = blockIdx.x;
    issue(0, tile);
    for (int stage = 0; tile < ntiles; tile += gridDim.x, stage ^= 1) {
        issue(stage ^ 1, tile + gridDim.x);                 // next tile in flight while this one computes
        ptx::cp_async_wait<1>();                            // this tile's copies (the older group) landed
        const long long i = tile * T + tid;
        if (i >= a.n) continue;
        const double* s = rls_ring + (static_cast<size_t>(stage) * NIN) * T + tid;
        double Y[M][P], z[M], th[P], C[P][P];
        int q = 0;
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int c = 0; c < P; ++c, ++q) Y[m][c] = s[q * T];
#pragma unroll
        for (int m = 0; m < M; ++m, ++q) z[m] = s[q * T];
#pragma unroll
        for (int c = 0; c < P; ++c, ++q) th[c] = s[q * T];
#pragma unroll
        for (int c = 0; c < P; ++c)
#pragma unroll
            for (int d = 0; d < P; ++d, ++q) C[c][d] = s[q * T];
        rls_advance<P, M>(Y, z, r, a.lambda, th, C);
#pragma unroll
        for (int c = 0; c < P; ++c) {
            __stcs(a.theta[c] + i, th[c]);
#pragma unroll
            for (int d = 0; d < P; ++d) __stcs(a.cov[c * P + d] + i, C[c][d]);
        }
    }
    ptx::cp_async_wait<0>();
}

// Fused: contact state -> regressor (registers) -> RLS update of (spring, damper) per contact.
// ------------------------------------------------------------------------------------------------
// General sizes and general S: the fallback of the register kernels above.
//
// The reference takes any number of parameters and measurements and inverts S = lambda R + Y P Y^T
// with Eigen's dynamic inverse(), i.e. an LU with partial pivoting -- it never requires S to be
// positive definite (src/Estimators/src/RecursiveLeastSquare.cpp:118-130).  The register kernels
// cover 1..4 x 1..6 and factorise S as LDL^T without pivoting, which presumes lambda R > 0.  This
// kernel does what the reference does, for any p, m: one estimator per thread, work arrays in a
// global scratch laid out [slot][estimator] (coalesced), the reference's association
//   K = (P Y^T) S^-1,  theta += K (z - Y theta),  P = (P - (K Y) P) / lambda
// and S^-1 by partial-pivot LU + n solves.  Not tuned: it exists so that nothing the reference
// accepts is refused (a singular S gives inf/NaN, as the reference).
// Arrays are array-of-structures (tabs == nullptr) or SoA planes through a device pointer table
// tabs = [Y planes m*p | z planes m | theta planes p | cov planes p*p].
// ------------------------------------------------------------------------------------------------
struct RlsGenArgs {
    const double* const* tabs;
    const double* Y;
    const double* z;
    double* theta;
    double* cov;
    const double* lr;      // device, m entries: lambda * r[i]
    double* work;          // rls_gen_work_doubles(p, m) * n doubles
    double lambda;
    long long n;
    int p, m;
};

__host__ __device__ inline long long rls_gen_work_doubles(int p, int m)
{
    // YP m*p | LU m*m | Sinv m*m | PYt p*m | K p*m | innov m | y m | perm m | KY p*p | Pnew p*p
    return 3LL * m * p + 2LL * m * m + 3LL * m + 2LL * p * p;
}

__global__ void __launch_bounds__(64)
rls_advance_generic_kernel(const __grid_constant__ RlsGenArgs a)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const int p = a.p, m = a.m;
    const long long n = a.n;
    const bool soa = a.tabs != nullptr;
    auto Yel = [&](int r, int c) { return soa ? a.tabs[r * p + c][i] : a.Y[i * m * p + r * p + c]; };
    auto zel = [&](int r) { return soa ? a.tabs[m * p + r][i] : a.z[i * m + r]; };
    auto thp = [&](int r) -> double* {
        return soa ? const_cast<double*>(a.tabs[m * p + m + r]) + i : a.theta + i * p + r;
    };
    auto Pp = [&](int r, int c) -> double* {
        return soa ? const_cast<double*>(a.tabs[m * p + m + p + r * p + c]) + i : a.cov + i * p * p + r * p + c;
    };
    double* w = a.work + i;
    auto W = [&](long long slot) -> double& { return w[slot * n]; };
    const long long oYP = 0, oLU = oYP + 1LL * m * p, oSI = oLU + 1LL * m * m, oPY = oSI + 1LL * m * m,
                    oK = oPY + 1LL * p * m, oIN = oK + 1LL * p * m, oY = oIN + m, oPM = oY + m,
                    oKY = oPM + m, oPN = oKY + 1LL * p * p;

    // YP = Y P ; S = lambda R + (Y P) Y^T
    for (int r = 0; r < m; ++r)
        for (int c = 0; c < p; ++c) {
            double acc = 0.0;
            for (int k = 0; k < p; ++k) acc = acc + Yel(r, k) * *Pp(k, c);
            W(oYP + r * p + c) = acc;
        }
    for (int r = 0; r < m; ++r)
        for (int c = 0; c < m; ++c) {
            double acc = 0.0;
            for (int k = 0; k < p; ++k) acc = acc + W(oYP + r * p + k) * Yel(c, k);
            W(oLU + r * m + c) = (r == c ? a.lr[r] : 0.0) + acc;
        }
    // LU with partial pivoting, in place; perm as doubles
    for (int r = 0; r < m; ++r) W(oPM + r) = r;
    for (int k = 0; k < m; ++k) {
        int piv = k;
        double best = fabs(W(oLU + k * m + k));
        for (int r = k + 1; r < m; ++r) {
            const double v = fabs(W(oLU + r * m + k));
            if (v > best) {
                best = v;
                piv = r;
            }
        }
        if (piv != k) {
            for (int c = 0; c < m; ++c) {
                const double t = W(oLU + k * m + c);
                W(oLU + k * m + c) = W(oLU + piv * m + c);
                W(oLU + piv * m + c) = t;
            }
            const double t = W(oPM + k);
            W(oPM + k) = W(oPM + piv);
            W(oPM + piv) = t;
        }
        const double d = W(oLU + k * m + k);
        for (int r = k + 1; r < m; ++r) {
            const double l = W(oLU + r * m + k) / d;
            W(oLU + r * m + k) = l;
            for (int c = k + 1; c < m; ++c) W(oLU + r * m + c) = W(oLU + r * m + c) - l * W(oLU + k * m + c);
        }
    }
    // Sinv: solve S x = e_c for every column
    for (int c = 0; c < m; ++c) {
        for (int r = 0; r < m; ++r) {
            double acc = (static_cast<int>(W(oPM + r)) == c) ? 1.0 : 0.0;
            for (int k = 0; k < r; ++k) acc = acc - W(oLU + r * m + k) * W(oY + k);
            W(oY + r) = acc;
        }
        for (int r = m - 1; r >= 0; --r) {
            double acc = W(oY + r);
            for (int k = r + 1; k < m; ++k) acc = acc - W(oLU + r * m + k) * W(oSI + k * m + c);
            W(oSI + r * m + c) = acc / W(oLU + r * m + r);
        }
    }
    // K = (P Y^T) S^-1
    for (int r = 0; r < p; ++r)
        for (int c = 0; c < m; ++c) {
            double acc = 0.0;
            for (int k = 0; k < p; ++k) acc = acc + *Pp(r, k) * Yel(c, k);
            W(oPY + r * m + c) = acc;
        }
    for (int r = 0; r < p; ++r)
        for (int c = 0; c < m; ++c) {
            double acc = 0.0;
            for (int k = 0; k < m; ++k) acc = acc + W(oPY + r * m + k) * W(oSI + k * m + c);
            W(oK + r * m + c) = acc;
        }
    // theta = theta + K (z - Y theta)
    for (int r = 0; r < m; ++r) {
        double acc = 0.0;
        for (int k = 0; k < p; ++k) acc = acc + Yel(r, k) * *thp(k);
        W(oIN + r) = zel(r) - acc;
    }
    for (int r = 0; r < p; ++r) {
        double acc = 0.0;
        for (int k = 0; k < m; ++k) acc = acc + W(oK + r * m + k) * W(oIN + k);
        *thp(r) = *thp(r) + acc;
    }
    // P = (P - (K Y) P) / lambda
    for (int r = 0; r < p; ++r)
        for (int c = 0; c < p; ++c) {
            double acc = 0.0;
            for (int k = 0; k < m; ++k) acc = acc + W(oK + r * m + k) * Yel(k, c);
            W(oKY + r * p + c) = acc;
        }
    for (int r = 0; r < p; ++r)
        for (int c = 0; c < p; ++c) {
            double acc = 0.0;
            for (int k = 0; k < p; ++k) acc = acc + W(oKY + r * p + k) * *Pp(k, c);
            W(oPN + r * p + c) = (*Pp(r, c) - acc) / a.lambda;
        }
    for (int r = 0; r < p; ++r)
        for (int c = 0; c < p; ++c) *Pp(r, c) = W(oPN + r * p + c);
}

struct CcmRlsArgs {
    const double* in[30];
    const double* geom[2];     // length, width planes (HETG) else uniform
    const double* z[6];        // measured wrench planes
    double* theta[2];          // spring, damper estimates (in/out)
    double* cov[4];            // 2x2 covariance, row-major planes (in/out)
    double w[6];               // lambda * r[i]
    double lambda;
    double length, width;
    long long n;
};

template <bool HETG>
__global__ void __launch_bounds__(128, 4)
ccm_rls_kernel(const __grid_constant__ CcmRlsArgs a)
{
    constexpr unsigned LIVE = live_planes(M_REGRESSOR);
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    double x[30] = {};
    load_live_planes<LIVE>(a.in, i, true, x);
    double z[6], r[6], th[2], C[2][2];
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        z[q] = __ldcs(a.z[q] + i);
        r[q] = a.w[q];
    }
    th[0] = __ldcs(a.theta[0] + i);
    th[1] = __ldcs(a.theta[1] + i);
    C[0][0] = __ldcs(a.cov[0] + i); C[0][1] = __ldcs(a.cov[1] + i);
    C[1][0] = __ldcs(a.cov[2] + i); C[1][1] = __ldcs(a.cov[3] + i);
    double L = a.length, W = a.width;
    if constexpr (HETG) {
        L = __ldcs(a.geom[0] + i);
        W = __ldcs(a.geom[1] + i);
    }
    Result res;
    eval_contact<M_REGRESSOR>(state_from_planes(x), make_prm(L, W, 0.0, 0.0), res);
    const double Y[6][2] = {{res.y_fk.x, res.y_fb.x}, {res.y_fk.y, res.y_fb.y}, {res.y_fk.z, res.y_fb.z},
                            {res.y_tk.x, res.y_tb.x}, {res.y_tk.y, res.y_tb.y}, {res.y_tk.z, res.y_tb.z}};
    rls_advance<2, 6>(Y, z, r, a.lambda, th, C);
    __stcs(a.theta[0] + i, th[0]);
    __stcs(a.theta[1] + i, th[1]);
    __stcs(a.cov[0] + i, C[0][0]); __stcs(a.cov[1] + i, C[0][1]);
    __stcs(a.cov[2] + i, C[1][0]); __stcs(a.cov[3] + i, C[1][1]);
}

}  // namespace blfccm
