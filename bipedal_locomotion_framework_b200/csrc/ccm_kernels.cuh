// ccm_kernels.cuh -- sm_100a kernels for batched ContinuousContactModel evaluation.
//
// Work decomposition (all kernels): a WARP owns a tile of 32 consecutive contacts and never
// synchronises with other warps.  Launches are one tile per warp (no persistent loop): measured on
// B200, the hardware CTA scheduler's natural staggering of loads and stores beats a persistent grid
// whose warps march in lock-step (profiles/r01_variant_sweep.md).  HBM streams are touched once:
//   SoA planes      coalesced 64-bit streaming loads / stores, one contact per lane (256 B per warp
//                   request = two full 128 B lines; LDG.E.EF.64 / STG.E.EF.64).  A 128-bit,
//                   two-contacts-per-lane variant was measured slower on B200 (its 166 registers
//                   cap occupancy at 12 warps/SM) and removed (DESIGN §5);
//   dense 6x6 ctrl  assembled per warp in shared memory, then ONE bulk async copy (TMA engine,
//                   SASS UBLKCP) of tile*288 contiguous bytes;
//   AoS structs     every input array arrives with a bulk async copy per tile signalled on a
//                   per-warp mbarrier; lanes pick their own struct out of shared memory
//                   (the AoS->SoA transposition); outputs leave through bulk stores too.
// FP64 arithmetic is in ccm_math.cuh.
#pragma once

#include "ccm_math.cuh"
#include "ccm_ptx.cuh"

namespace blfccm {

constexpr int kWarp = 32;

__device__ __forceinline__ long long min64(long long a, long long b) { return a < b ? a : b; }

// ------------------------------------------------------------------------------------------------
// SoA kernels
// ------------------------------------------------------------------------------------------------

struct SoaArgs {
    const double* in[30];
    const double* prm[4];      // length, width, spring, damper planes (HET only)
    double* wrench[6];
    double* autodyn[6];
    double* reg[12];
    double* ctrl;
    Prm uni;
    long long n;
    int ctrl_bulk;             // ctrl is 16-byte aligned -> bulk store
    // sampling-MPC cost epilogue (COST kernels only)
    long long rollout_len;
    double ref[6];             // reference wrench
    double wf, wt;             // force / torque weights
    double* partials;          // [n_rollouts][slots] per-(rollout, tile) partial sums
    int slots;                 // max tiles one rollout can intersect
};

// write the 12 non-structural entries of one dense 6x6 into its slot of the warp's tile
__device__ __forceinline__ void stage_ctrl(double* slot, const Result& r)
{
    slot[0] = r.gd;
    slot[7] = r.gd;
    slot[14] = r.gd;
    slot[21] = r.gs[0];
    *reinterpret_cast<double2*>(slot + 22) = make_double2(r.gs[1], r.gs[2]);
    slot[27] = r.gs[1];
    *reinterpret_cast<double2*>(slot + 28) = make_double2(r.gs[3], r.gs[4]);
    slot[33] = r.gs[2];
    *reinterpret_cast<double2*>(slot + 34) = make_double2(r.gs[4], r.gs[5]);
}

// flush `cnt` staged 6x6 blocks (contiguous in shared memory) to ctrl + base*36
__device__ __forceinline__ void flush_ctrl_tile(double* __restrict__ ctrl, const double* tile,
                                                long long base, int cnt, int lane, bool bulk)
{
    if (bulk) {
        ptx::fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            ptx::bulk_s2g(ctrl + base * 36, ptx::smem_addr(tile), static_cast<uint32_t>(cnt) * 288u);
            ptx::bulk_commit();
        }
    } else {
        __syncwarp();
        for (int i = lane; i < cnt * 36; i += kWarp) __stcs(ctrl + base * 36 + i, tile[i]);
    }
}

// first tile (of 32 contacts) a rollout touches, and its slot for tile t
__device__ __forceinline__ long long rollout_first_tile(long long rid, long long len)
{
    return (rid * len) >> 5;
}

// Primary kernel: one contact per lane, one 32-contact tile per warp, no loop.
//   OUT   outputs written to HBM (bits of the C-ABI out_mask)
//   COST  also reduce  wf|F-Fref|^2 + wt|T-Tref|^2  per (rollout, tile) into a.partials
//         (fixed-order butterfly: deterministic); the wrench is then computed even if not in OUT.
template <unsigned OUT, bool HET, bool COST>
__global__ void __launch_bounds__(128, ((OUT & M_CTRL) ? 5 : 6))
ccm_soa_kernel(const __grid_constant__ SoaArgs a)
{
    constexpr unsigned MASK = OUT | (COST ? M_WRENCH : 0u);
    constexpr unsigned LIVE = live_planes(MASK);
    extern __shared__ __align__(128) unsigned char smem_raw[];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long tile = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + warp;
    const long long base = tile << 5;
    if (base >= a.n) return;  // warp-uniform
    const long long i = base + lane;
    const bool on = i < a.n;
    const int cnt = static_cast<int>(min64(kWarp, a.n - base));

    // Programmatic dependent launch: let the NEXT launch of the stream take SM slots as this grid's
    // CTAs retire; such a CTA does the part of its work that touches no global memory (the
    // structural zeros below) and then blocks in grid_dep_wait() until the previous grid has
    // completed -- stream order is preserved, the inter-launch gap and the ramp of the first wave
    // disappear.  (Without the launch attribute both instructions are no-ops.)
    ptx::grid_dep_launch_dependents();

    double* ctile = reinterpret_cast<double*>(smem_raw) + warp * (kWarp * 36);
    if constexpr ((OUT & M_CTRL) != 0) {
        // structural zeros of the 32 dense blocks
        double2* z = reinterpret_cast<double2*>(ctile);
#pragma unroll
        for (int j = 0; j < 18; ++j) z[lane + j * kWarp] = make_double2(0.0, 0.0);
        __syncwarp();
    }
    ptx::grid_dep_wait();

    // ---- every live plane in flight before the first use ---------------------------------------
    double x[30] = {};
    load_live_planes<LIVE>(a.in, i, on, x);
    const Prm q = load_params<HET>(a.prm, a.uni, i, on);
    Result r;
    eval_contact<MASK>(state_from_planes(x), q, r);

    if (on) {
        if constexpr ((OUT & M_WRENCH) != 0) store_wrench(a.wrench, i, r);
        if constexpr ((OUT & M_AUTODYN) != 0) {
            __stcs(a.autodyn[0] + i, r.fhead.x); __stcs(a.autodyn[1] + i, r.fhead.y);
            __stcs(a.autodyn[2] + i, r.fhead.z); __stcs(a.autodyn[3] + i, r.ftail.x);
            __stcs(a.autodyn[4] + i, r.ftail.y); __stcs(a.autodyn[5] + i, r.ftail.z);
        }
        if constexpr ((OUT & M_REGRESSOR) != 0) {
            // row-major 6x2: plane 2*row + col, col 0 = spring, col 1 = damper
            __stcs(a.reg[0] + i, r.y_fk.x); __stcs(a.reg[1] + i, r.y_fb.x);
            __stcs(a.reg[2] + i, r.y_fk.y); __stcs(a.reg[3] + i, r.y_fb.y);
            __stcs(a.reg[4] + i, r.y_fk.z); __stcs(a.reg[5] + i, r.y_fb.z);
            __stcs(a.reg[6] + i, r.y_tk.x); __stcs(a.reg[7] + i, r.y_tb.x);
            __stcs(a.reg[8] + i, r.y_tk.y); __stcs(a.reg[9] + i, r.y_tb.y);
            __stcs(a.reg[10] + i, r.y_tk.z); __stcs(a.reg[11] + i, r.y_tb.z);
        }
        if constexpr ((OUT & M_CTRL) != 0) stage_ctrl(ctile + lane * 36, r);
    }
    if constexpr ((OUT & M_CTRL) != 0) flush_ctrl_tile(a.ctrl, ctile, base, cnt, lane, a.ctrl_bulk != 0);

    if constexpr (COST) {
        double c = 0.0;
        if (on) {
            const V3 df = r.force - V3{a.ref[0], a.ref[1], a.ref[2]};
            const V3 dt = r.torque - V3{a.ref[3], a.ref[4], a.ref[5]};
            c = a.wf * (df.x * df.x + df.y * df.y + df.z * df.z) +
                a.wt * (dt.x * dt.x + dt.y * dt.y + dt.z * dt.z);
        }
        const long long rid = (on ? i : base + cnt - 1) / a.rollout_len;
        const long long rid_first = __shfl_sync(0xffffffffu, rid, 0);
        const long long rid_last = __shfl_sync(0xffffffffu, rid, cnt - 1);
        for (long long rr = rid_first; rr <= rid_last; ++rr) {
            double v = (on && rid == rr) ? c : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0)
                a.partials[rr * a.slots + (tile - rollout_first_tile(rr, a.rollout_len))] = v;
        }
    }

    if constexpr ((OUT & M_CTRL) != 0) {
        // shared memory must stay valid until the bulk engine has read it
        if (a.ctrl_bulk && lane == 0) ptx::bulk_wait_read_all();
    }
}

// ------------------------------------------------------------------------------------------------
// AoS kernel (bulk-copy staged; every pointer 16-byte aligned)
// ------------------------------------------------------------------------------------------------

struct AosArgs {
    const double* twists;      // n*6
    const double* poses;       // n*12
    const double* nulls;       // n*12
    const double* prm;         // n*4 (HET only)
    double* wrench;            // n*6
    double* autodyn;           // n*6
    double* ctrl;              // n*36
    double* reg;               // n*12
    Prm uni;
    long long n;
    int ctrl_compact;          // ctrl receives n*8 doubles {gd, gs[0..5], 0} instead of n*36 (host pipeline)
};

// the 7 distinct values of one control matrix, padded to 8 doubles
__device__ __forceinline__ void stage_ctrl_compact(double* slot, const Result& r)
{
    double2* o = reinterpret_cast<double2*>(slot);
    o[0] = make_double2(r.gd, r.gs[0]);
    o[1] = make_double2(r.gs[1], r.gs[2]);
    o[2] = make_double2(r.gs[3], r.gs[4]);
    o[3] = make_double2(r.gs[5], 0.0);
}

// per-warp shared-memory layout for a 32-contact tile (byte offsets, all multiples of 128)
template <unsigned MASK, bool HET>
struct AosSmem {
    static constexpr bool kNeedState = (MASK & (M_WRENCH | M_AUTODYN | M_REGRESSOR)) != 0;
    static constexpr int tw = 0;                                       // 32*48
    static constexpr int po = tw + (kNeedState ? 1536 : 0);            // 32*96
    static constexpr int nu = po + 3072;                               // 32*96
    static constexpr int pr = nu + (kNeedState ? 3072 : 0);            // 32*32
    static constexpr int ow = pr + (HET ? 1024 : 0);                   // 32*48
    static constexpr int oa = ow + ((MASK & M_WRENCH) ? 1536 : 0);     // 32*48
    static constexpr int og = oa + ((MASK & M_AUTODYN) ? 1536 : 0);    // 32*96
    static constexpr int oc = og + ((MASK & M_REGRESSOR) ? 3072 : 0);  // 32*288
    static constexpr int bar = oc + ((MASK & M_CTRL) ? 9216 : 0);
    static constexpr int bytes = bar + 128;
    static constexpr uint32_t in_bytes_per_contact =
        (kNeedState ? 48u + 96u : 0u) + 96u + (HET ? 32u : 0u);
};

template <unsigned MASK, bool HET>
__device__ __forceinline__ void aos_issue_loads(const AosArgs& a, unsigned char* ws, uint32_t bar,
                                                long long base, int cnt)
{
    using S = AosSmem<MASK, HET>;
    const uint32_t c = static_cast<uint32_t>(cnt);
    ptx::mbar_arrive_expect_tx(bar, c * S::in_bytes_per_contact);
    if constexpr (S::kNeedState) {
        ptx::bulk_g2s(ptx::smem_addr(ws + S::tw), a.twists + base * 6, c * 48u, bar);
        ptx::bulk_g2s(ptx::smem_addr(ws + S::nu), a.nulls + base * 12, c * 96u, bar);
    }
    ptx::bulk_g2s(ptx::smem_addr(ws + S::po), a.poses + base * 12, c * 96u, bar);
    if constexpr (HET) ptx::bulk_g2s(ptx::smem_addr(ws + S::pr), a.prm + base * 4, c * 32u, bar);
}

template <unsigned MASK, bool HET>
__global__ void __launch_bounds__(64)
ccm_aos_kernel(const __grid_constant__ AosArgs a)
{
    using S = AosSmem<MASK, HET>;
    constexpr int TILE = kWarp;
    extern __shared__ __align__(128) unsigned char smem_raw[];

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int warps_per_cta = blockDim.x >> 5;
    unsigned char* ws = smem_raw + static_cast<size_t>(warp) * S::bytes;
    const uint32_t bar = ptx::smem_addr(ws + S::bar);

    if (lane == 0) {
        ptx::mbar_init(bar, 1);
        ptx::fence_mbar_init();
    }
    if constexpr ((MASK & M_CTRL) != 0) {
        double2* z = reinterpret_cast<double2*>(ws + S::oc);
        for (int i = lane; i < TILE * 18; i += kWarp) z[i] = make_double2(0.0, 0.0);
    }
    __syncwarp();
    ptx::grid_dep_launch_dependents();   // PDL: see ccm_soa_kernel
    ptx::grid_dep_wait();

    const long long ntiles = (a.n + TILE - 1) / TILE;
    const long long wstride = static_cast<long long>(gridDim.x) * warps_per_cta;
    long long t = static_cast<long long>(blockIdx.x) * warps_per_cta + warp;
    uint32_t phase = 0;

    if (t < ntiles && lane == 0) {
        const long long base = t * TILE;
        aos_issue_loads<MASK, HET>(a, ws, bar, base,
                                   static_cast<int>(min64(TILE, a.n - base)));
    }
    for (; t < ntiles; t += wstride) {
        const long long base = t * TILE;
        const int cnt = static_cast<int>(min64(TILE, a.n - base));
        const bool mine = lane < cnt;

        ptx::mbar_wait(bar, phase);
        phase ^= 1u;

        // ---- AoS -> registers: each lane lifts its own structs out of the staged tile -------
        State s;
        s.R02 = s.R12 = 0.0;
        Prm q = a.uni;
        {
            const double2* P = reinterpret_cast<const double2*>(ws + S::po) + lane * 6;
            const double2 p01 = P[0], p2r0 = P[1], r12 = P[2], r34 = P[3], r56 = P[4], r78 = P[5];
            // pose = px py | pz R00 | R01 R02 | R10 R11 | R12 R20 | R21 R22
            s.p = V3{p01.x, p01.y, p2r0.x};
            s.e1 = V3{p2r0.y, r34.x, r56.y};
            s.e2 = V3{r12.x, r34.y, r78.x};
            s.R02 = r12.y;
            s.R12 = r56.x;
            s.R22 = r78.y;
        }
        if constexpr (S::kNeedState) {
            const double2* T = reinterpret_cast<const double2*>(ws + S::tw) + lane * 3;
            const double2 t01 = T[0], t23 = T[1], t45 = T[2];
            s.v = V3{t01.x, t01.y, t23.x};
            s.w = V3{t23.y, t45.x, t45.y};
            const double2* N = reinterpret_cast<const double2*>(ws + S::nu) + lane * 6;
            const double2 n01 = N[0], n2r0 = N[1], m12 = N[2], m34 = N[3], m56 = N[4], m78 = N[5];
            s.p0 = V3{n01.x, n01.y, n2r0.x};
            s.n1 = V3{n2r0.y, m34.x, m56.y};
            s.n2 = V3{m12.x, m34.y, m78.x};
        }
        if constexpr (HET) {
            const double2* Q = reinterpret_cast<const double2*>(ws + S::pr) + lane * 2;
            const double2 lw = Q[0], kb = Q[1];
            q = make_prm(lw.x, lw.y, kb.x, kb.y);
        }
        __syncwarp();  // every lane has its inputs in registers: the stage is free again

        // ---- prefetch the next tile while this one is computed ------------------------------
        if (lane == 0) {
            const long long tn = t + wstride;
            if (tn < ntiles) {
                const long long bn = tn * TILE;
                aos_issue_loads<MASK, HET>(a, ws, bar, bn,
                                           static_cast<int>(min64(TILE, a.n - bn)));
            }
        }

        Result r;
        eval_contact<MASK>(s, q, r);

        // ---- outputs: stage in shared memory, leave through bulk stores ---------------------
        if (lane == 0) ptx::bulk_wait_read_all();
        __syncwarp();
        if (mine) {
            if constexpr ((MASK & M_WRENCH) != 0) {
                double2* o = reinterpret_cast<double2*>(ws + S::ow) + lane * 3;
                o[0] = make_double2(r.force.x, r.force.y);
                o[1] = make_double2(r.force.z, r.torque.x);
                o[2] = make_double2(r.torque.y, r.torque.z);
            }
            if constexpr ((MASK & M_AUTODYN) != 0) {
                double2* o = reinterpret_cast<double2*>(ws + S::oa) + lane * 3;
                o[0] = make_double2(r.fhead.x, r.fhead.y);
                o[1] = make_double2(r.fhead.z, r.ftail.x);
                o[2] = make_double2(r.ftail.y, r.ftail.z);
            }
            if constexpr ((MASK & M_REGRESSOR) != 0) {
                double2* o = reinterpret_cast<double2*>(ws + S::og) + lane * 6;
                o[0] = make_double2(r.y_fk.x, r.y_fb.x);
                o[1] = make_double2(r.y_fk.y, r.y_fb.y);
                o[2] = make_double2(r.y_fk.z, r.y_fb.z);
                o[3] = make_double2(r.y_tk.x, r.y_tb.x);
                o[4] = make_double2(r.y_tk.y, r.y_tb.y);
                o[5] = make_double2(r.y_tk.z, r.y_tb.z);
            }
            if constexpr ((MASK & M_CTRL) != 0) {
                if (a.ctrl_compact) stage_ctrl_compact(reinterpret_cast<double*>(ws + S::oc) + lane * 8, r);
                else stage_ctrl(reinterpret_cast<double*>(ws + S::oc) + lane * 36, r);
            }
        }
        ptx::fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            const uint32_t c = static_cast<uint32_t>(cnt);
            if constexpr ((MASK & M_WRENCH) != 0)
                ptx::bulk_s2g(a.wrench + base * 6, ptx::smem_addr(ws + S::ow), c * 48u);
            if constexpr ((MASK & M_AUTODYN) != 0)
                ptx::bulk_s2g(a.autodyn + base * 6, ptx::smem_addr(ws + S::oa), c * 48u);
            if constexpr ((MASK & M_REGRESSOR) != 0)
                ptx::bulk_s2g(a.reg + base * 12, ptx::smem_addr(ws + S::og), c * 96u);
            if constexpr ((MASK & M_CTRL) != 0) {
                if (a.ctrl_compact) ptx::bulk_s2g(a.ctrl + base * 8, ptx::smem_addr(ws + S::oc), c * 64u);
                else ptx::bulk_s2g(a.ctrl + base * 36, ptx::smem_addr(ws + S::oc), c * 288u);
            }
            ptx::bulk_commit();
        }
    }
    if (lane == 0) ptx::bulk_wait_all();
}

// ------------------------------------------------------------------------------------------------
// AoS kernel for buffers that are only 8-byte aligned: direct 64-bit loads/stores per lane.
// Same arithmetic, no staging; the checked (not silent) slow path of the C ABI.
// ------------------------------------------------------------------------------------------------

template <unsigned MASK, bool HET>
__global__ void __launch_bounds__(128)
ccm_aos_scalar_kernel(const __grid_constant__ AosArgs a)
{
    constexpr bool kNeedState = (MASK & (M_WRENCH | M_AUTODYN | M_REGRESSOR)) != 0;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.n;
         i += stride) {
        State s;
        const double* P = a.poses + i * 12;
        s.p = V3{P[0], P[1], P[2]};
        s.e1 = V3{P[3], P[6], P[9]};
        s.e2 = V3{P[4], P[7], P[10]};
        s.R02 = P[5];
        s.R12 = P[8];
        s.R22 = P[11];
        if constexpr (kNeedState) {
            const double* T = a.twists + i * 6;
            s.v = V3{T[0], T[1], T[2]};
            s.w = V3{T[3], T[4], T[5]};
            const double* N = a.nulls + i * 12;
            s.p0 = V3{N[0], N[1], N[2]};
            s.n1 = V3{N[3], N[6], N[9]};
            s.n2 = V3{N[4], N[7], N[10]};
        }
        Prm q = a.uni;
        if constexpr (HET) {
            const double* Q = a.prm + i * 4;
            q = make_prm(Q[0], Q[1], Q[2], Q[3]);
        }
        Result r;
        eval_contact<MASK>(s, q, r);
        if constexpr ((MASK & M_WRENCH) != 0) {
            double* o = a.wrench + i * 6;
            o[0] = r.force.x; o[1] = r.force.y; o[2] = r.force.z;
            o[3] = r.torque.x; o[4] = r.torque.y; o[5] = r.torque.z;
        }
        if constexpr ((MASK & M_AUTODYN) != 0) {
            double* o = a.autodyn + i * 6;
            o[0] = r.fhead.x; o[1] = r.fhead.y; o[2] = r.fhead.z;
            o[3] = r.ftail.x; o[4] = r.ftail.y; o[5] = r.ftail.z;
        }
        if constexpr ((MASK & M_REGRESSOR) != 0) {
            double* o = a.reg + i * 12;
            o[0] = r.y_fk.x; o[1] = r.y_fb.x; o[2] = r.y_fk.y; o[3] = r.y_fb.y;
            o[4] = r.y_fk.z; o[5] = r.y_fb.z; o[6] = r.y_tk.x; o[7] = r.y_tb.x;
            o[8] = r.y_tk.y; o[9] = r.y_tb.y; o[10] = r.y_tk.z; o[11] = r.y_tb.z;
        }
        if constexpr ((MASK & M_CTRL) != 0) {
            if (a.ctrl_compact) {
                double* o = a.ctrl + i * 8;
                o[0] = r.gd;
#pragma unroll
                for (int e = 0; e < 6; ++e) o[1 + e] = r.gs[e];
                o[7] = 0.0;
                continue;
            }
            double* o = a.ctrl + i * 36;
#pragma unroll
            for (int e = 0; e < 36; ++e) o[e] = 0.0;
            o[0] = r.gd; o[7] = r.gd; o[14] = r.gd;
            o[21] = r.gs[0]; o[22] = r.gs[1]; o[23] = r.gs[2];
            o[27] = r.gs[1]; o[28] = r.gs[3]; o[29] = r.gs[4];
            o[33] = r.gs[2]; o[34] = r.gs[4]; o[35] = r.gs[5];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// One contact state (the per-instance facade's getters): the state travels in the kernel
// parameters, the results go straight to mapped pinned host memory -- one launch and one stream
// synchronisation per getter instead of three staged copies around a batch kernel.
// ------------------------------------------------------------------------------------------------

struct SingleArgs {
    double tw[6];
    double pose[12];
    double null[12];
    Prm prm;
    double* out;   // mapped host memory: wrench 0-5 | autodyn 6-11 | regressor 12-23 | ctrl 24-59 | flag 60
    unsigned long long seq;   // written to out[60] after the results: the host polls it
};

template <unsigned MASK>
__global__ void ccm_single_kernel(const __grid_constant__ SingleArgs a)
{
    if (threadIdx.x != 0) return;
    State s;
    s.v = V3{a.tw[0], a.tw[1], a.tw[2]};
    s.w = V3{a.tw[3], a.tw[4], a.tw[5]};
    s.p = V3{a.pose[0], a.pose[1], a.pose[2]};
    s.e1 = V3{a.pose[3], a.pose[6], a.pose[9]};
    s.e2 = V3{a.pose[4], a.pose[7], a.pose[10]};
    s.R02 = a.pose[5];
    s.R12 = a.pose[8];
    s.R22 = a.pose[11];
    s.p0 = V3{a.null[0], a.null[1], a.null[2]};
    s.n1 = V3{a.null[3], a.null[6], a.null[9]};
    s.n2 = V3{a.null[4], a.null[7], a.null[10]};
    Result r;
    eval_contact<MASK>(s, a.prm, r);
    double* o = a.out;
    if constexpr ((MASK & M_WRENCH) != 0) {
        o[0] = r.force.x; o[1] = r.force.y; o[2] = r.force.z;
        o[3] = r.torque.x; o[4] = r.torque.y; o[5] = r.torque.z;
    }
    if constexpr ((MASK & M_AUTODYN) != 0) {
        o[6] = r.fhead.x; o[7] = r.fhead.y; o[8] = r.fhead.z;
        o[9] = r.ftail.x; o[10] = r.ftail.y; o[11] = r.ftail.z;
    }
    if constexpr ((MASK & M_REGRESSOR) != 0) {
        o[12] = r.y_fk.x; o[13] = r.y_fb.x; o[14] = r.y_fk.y; o[15] = r.y_fb.y;
        o[16] = r.y_fk.z; o[17] = r.y_fb.z; o[18] = r.y_tk.x; o[19] = r.y_tb.x;
        o[20] = r.y_tk.y; o[21] = r.y_tb.y; o[22] = r.y_tk.z; o[23] = r.y_tb.z;
    }
    if constexpr ((MASK & M_CTRL) != 0) {
        double* c = o + 24;
#pragma unroll
        for (int e = 0; e < 36; ++e) c[e] = 0.0;
        c[0] = r.gd; c[7] = r.gd; c[14] = r.gd;
        c[21] = r.gs[0]; c[22] = r.gs[1]; c[23] = r.gs[2];
        c[27] = r.gs[1]; c[28] = r.gs[3]; c[29] = r.gs[4];
        c[33] = r.gs[2]; c[34] = r.gs[4]; c[35] = r.gs[5];
    }
    // results first, then the sequence number: the host spins on it instead of paying a stream
    // synchronisation per getter
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(o + 60) = a.seq;
}

// ------------------------------------------------------------------------------------------------
// Surface points of one contact state (getForceAtPoint / getTorqueGeneratedAtPoint)
// ------------------------------------------------------------------------------------------------

struct PointArgs {
    double tw[6];
    double pose[12];
    double null[12];
    double length, width, k, b;
    const double* xy;
    double* force;
    double* torque;
    long long m;
};

__global__ void __launch_bounds__(128)
ccm_surface_points_kernel(const __grid_constant__ PointArgs a)
{
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    const V3 v{a.tw[0], a.tw[1], a.tw[2]}, w{a.tw[3], a.tw[4], a.tw[5]};
    const V3 p{a.pose[0], a.pose[1], a.pose[2]}, p0{a.null[0], a.null[1], a.null[2]};
    const V3 e1{a.pose[3], a.pose[6], a.pose[9]}, e2{a.pose[4], a.pose[7], a.pose[10]};
    const V3 n1{a.null[3], a.null[6], a.null[9]}, n2{a.null[4], a.null[7], a.null[10]};
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < a.m;
         i += stride) {
        const double x = a.xy[2 * i], y = a.xy[2 * i + 1];
        V3 f{0.0, 0.0, 0.0}, tq{0.0, 0.0, 0.0};
        // ContinuousContactModel.cpp:185-189 (strict >: the boundary is inside)
        if (!(fabs(x) > a.length / 2 || fabs(y) > a.width / 2)) {
            const V3 rq = x * e1 + y * e2;                 // R q,  q = (x, y, 0)
            const V3 r0q = x * n1 + y * n2;                // R0 q
            // k((p0 - p) + (R0 - R) q) - b(v + w x (R q))        :196-199
            f = a.k * ((p0 - p) + (r0q - rq)) - a.b * (v + cross(w, rq));
            tq = cross(rq, f);                             // :219
        }
        if (a.force) {
            a.force[3 * i] = f.x; a.force[3 * i + 1] = f.y; a.force[3 * i + 2] = f.z;
        }
        if (a.torque) {
            a.torque[3 * i] = tq.x; a.torque[3 * i + 1] = tq.y; a.torque[3 * i + 2] = tq.z;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Sampling-MPC epilogue, second (tiny) launch: sum each rollout's per-tile partials in tile order,
// write cost[r], arg-min with lowest-index tie-break.  Device-wide arg-min by the last-block-done
// pattern: every CTA publishes its (cost,index) pair, the last one to finish combines them.
// ------------------------------------------------------------------------------------------------

struct CostIdx {
    double cost;
    long long idx;
};

__device__ __forceinline__ bool better(double c, long long i, double bc, long long bi)
{
    return (c < bc) || (c == bc && i < bi);
}

__device__ __forceinline__ CostIdx warp_best(CostIdx b)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double c = __shfl_xor_sync(0xffffffffu, b.cost, o);
        const long long i = __shfl_xor_sync(0xffffffffu, b.idx, o);
        if (better(c, i, b.cost, b.idx)) {
            b.cost = c;
            b.idx = i;
        }
    }
    return b;
}

// ------------------------------------------------------------------------------------------------
// Reverse mode of the wrench (vector-Jacobian product), organised as ccm_soa_kernel: one contact
// per lane, one 32-contact tile per warp, every live plane in flight before the first use,
// streaming 64-bit loads and stores.  GROUPS (G_TWIST | G_POSE | G_NULL | G_PARAMS) selects the
// gradients computed; only the input planes those need are read.
// ------------------------------------------------------------------------------------------------

struct VjpArgs {
    const double* in[30];
    const double* prm[4];      // length, width, spring, damper planes (HET only)
    const double* gw[6];       // cotangent planes gF, gT; nullptr = zero
    double* gin[30];           // gradient planes of the state; nullptr = not written
    double* gprm[4];           // per-contact gradient of length, width, spring, damper (G_PARAMS)
    double uni[4];             // uniform length, width, spring, damper
    long long n;
};

template <unsigned GROUPS, bool HET>
__global__ void __launch_bounds__(128)
ccm_wrench_vjp_kernel(const __grid_constant__ VjpArgs a)
{
    constexpr unsigned LIVE = vjp_live_planes(GROUPS);
    const int lane = threadIdx.x & 31;
    const long long tile = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long base = tile << 5;
    if (base >= a.n) return;  // warp-uniform
    const long long i = base + lane;
    const bool on = i < a.n;

    ptx::grid_dep_launch_dependents();
    ptx::grid_dep_wait();

    double x[30] = {};
    load_live_planes<LIVE>(a.in, i, on, x);
    double gw[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) gw[j] = (on && a.gw[j]) ? __ldcs(a.gw[j] + i) : 0.0;
    double l = a.uni[0], w = a.uni[1], k = a.uni[2], b = a.uni[3];
    if constexpr (HET) {
        l = on ? __ldcs(a.prm[0] + i) : 0.0;
        w = on ? __ldcs(a.prm[1] + i) : 0.0;
        k = on ? __ldcs(a.prm[2] + i) : 0.0;
        b = on ? __ldcs(a.prm[3] + i) : 0.0;
    }
    const Prm q = make_prm(l, w, k, b);

    VjpOut g;
    vjp_wrench<GROUPS>(state_from_planes(x), q, l, w, V3{gw[0], gw[1], gw[2]}, V3{gw[3], gw[4], gw[5]}, g);
    if (!on) return;

    auto put = [&](int pl, double val) {
        if (a.gin[pl]) __stcs(a.gin[pl] + i, val);
    };
    if constexpr ((GROUPS & G_TWIST) != 0) {
        put(0, g.v.x); put(1, g.v.y); put(2, g.v.z);
        put(3, g.w.x); put(4, g.w.y); put(5, g.w.z);
    }
    if constexpr ((GROUPS & G_POSE) != 0) {
        put(6, g.p.x); put(7, g.p.y); put(8, g.p.z);
        put(9, g.e1.x); put(10, g.e2.x); put(11, 0.0);
        put(12, g.e1.y); put(13, g.e2.y); put(14, 0.0);
        put(15, g.e1.z); put(16, g.e2.z); put(17, g.R22);
    }
    if constexpr ((GROUPS & G_NULL) != 0) {
        put(18, g.p0.x); put(19, g.p0.y); put(20, g.p0.z);
        put(21, g.n1.x); put(22, g.n2.x); put(23, 0.0);
        put(24, g.n1.y); put(25, g.n2.y); put(26, 0.0);
        put(27, g.n1.z); put(28, g.n2.z); put(29, 0.0);
    }
    if constexpr ((GROUPS & G_PARAMS) != 0) {
        __stcs(a.gprm[0] + i, g.L); __stcs(a.gprm[1] + i, g.W);
        __stcs(a.gprm[2] + i, g.k); __stcs(a.gprm[3] + i, g.b);
    }
}

}  // namespace blfccm
#include "p2p_kernels.cuh"
namespace blfccm {

struct ReduceArgs {
    const double* partials;    // [n_rollouts][slots]
    int slots;
    int fixed_count;           // > 0: every rollout has exactly this many partials (slots == it)
    long long n_rollouts;
    long long rollout_len;
    long long index_base;
    double* cost;              // n_rollouts or nullptr
    CostIdx* block_best;       // gridDim.x entries (handle scratch)
    unsigned int* counter;     // zero before launch; reset by the last CTA
    CostIdx* best;             // result
    P2pArgs p2p;               // nranks > 0: the last block also runs the peer exchange -> p2p.out
};

__global__ void __launch_bounds__(128)
ccm_cost_reduce_kernel(const __grid_constant__ ReduceArgs ra)
{
    __shared__ CostIdx s_best[4];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    ptx::grid_dep_launch_dependents();   // PDL: see ccm_soa_kernel
    ptx::grid_dep_wait();                // the partials come from the previous launch

    CostIdx mine{inf, 0x7fffffffffffffffLL};
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long ro = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
         ro < ra.n_rollouts; ro += stride) {
        long long cntp = ra.fixed_count;
        if (cntp <= 0) {
            const long long t0 = rollout_first_tile(ro, ra.rollout_len);
            const long long t1 = ((ro + 1) * ra.rollout_len - 1) >> 5;
            cntp = t1 - t0 + 1;
        }
        const double* p = ra.partials + ro * ra.slots;
        double acc = 0.0;
        for (long long j = 0; j < cntp; ++j) acc += p[j];
        if (ra.cost) ra.cost[ro] = acc;
        const long long gi = ra.index_base + ro;
        if (better(acc, gi, mine.cost, mine.idx)) {
            mine.cost = acc;
            mine.idx = gi;
        }
    }
    mine = warp_best(mine);
    if (lane == 0) s_best[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        CostIdx b = s_best[0];
        for (int w = 1; w < (blockDim.x >> 5); ++w)
            if (better(s_best[w].cost, s_best[w].idx, b.cost, b.idx)) b = s_best[w];
        ra.block_best[blockIdx.x] = b;
        __threadfence();
        const unsigned int done = atomicAdd(ra.counter, 1u);
        s_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && warp == 0) {
        __threadfence();
        CostIdx b{inf, 0x7fffffffffffffffLL};
        for (unsigned int j = lane; j < gridDim.x; j += kWarp) {
            CostIdx c;
            c.cost = *reinterpret_cast<volatile double*>(&ra.block_best[j].cost);
            c.idx = *reinterpret_cast<volatile long long*>(&ra.block_best[j].idx);
            if (better(c.cost, c.idx, b.cost, b.idx)) b = c;
        }
        b = warp_best(b);
        if (b.idx == 0x7fffffffffffffffLL) b.idx = -1;  // nothing comparable (empty / all NaN)
        if (lane == 0) {
            *ra.best = b;
            *ra.counter = 0u;
        }
        // fused collective: this rank's pair goes straight to the peers' mailboxes over NVLink
        if (ra.p2p.nranks > 0) {
            const CostIdx g = p2p_exchange_warp(ra.p2p, b, lane);
            if (lane == 0) *ra.p2p.out = g;
        }
    }
}

// combine n (cost,index) pairs, lowest index wins ties; one warp
__global__ void ccm_argmin_pairs_kernel(const CostIdx* pairs, int n, CostIdx* best)
{
    const int lane = threadIdx.x;
    CostIdx b{__longlong_as_double(0x7ff0000000000000LL), 0x7fffffffffffffffLL};
    for (int j = lane; j < n; j += kWarp) {
        const CostIdx c = pairs[j];
        if (c.idx >= 0 && better(c.cost, c.idx, b.cost, b.idx)) b = c;
    }
    b = warp_best(b);
    if (lane == 0) {
        if (b.idx == 0x7fffffffffffffffLL) b.idx = -1;
        *best = b;
    }
}

}  // namespace blfccm
