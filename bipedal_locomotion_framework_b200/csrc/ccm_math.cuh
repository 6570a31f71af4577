// ccm_math.cuh -- per-contact closed form of ContinuousContactModel, register-resident FP64.
//
// Mathematics follows the reference (src/ContactModels/src/ContinuousContactModel.cpp):
//   wrench     :79-108    autonomous dynamics :110-146    control matrix :148-171
//   regressor  :223-254   point force/torque  :173-221
// but is derived independently in cross-product form: S(a)b = a x b, S(e)S(e)w = e x (e x w),
// Rdot.col(i) = w x e_i, S(e)^2 = e e^T - |e|^2 I.  One evaluation shares every sub-expression
// across the four outputs (the reference recomputes them per getter).  The reference's sign quirk
// is kept: wrench and regressor use |R22|, autonomous dynamics and control matrix use signed R22.
//
// Everything here is plain FP64 FMA-pipe work (DFMA/DMUL/DADD); tensor cores do not apply to
// per-contact 3-vector algebra.
#pragma once

#include <cuda_runtime.h>

namespace blfccm {

enum : unsigned { M_WRENCH = 1u, M_AUTODYN = 2u, M_CTRL = 4u, M_REGRESSOR = 8u };

// Parameters of one contact, with the products every output needs.
struct Prm {
    double L2;    // length^2
    double W2;    // width^2
    double A;     // length*width
    double A12;   // length*width/12
    double k;     // spring_coeff
    double b;     // damper_coeff
};

__host__ __device__ __forceinline__ Prm make_prm(double length, double width, double k, double b)
{
    Prm p;
    p.L2 = length * length;
    p.W2 = width * width;
    p.A = length * width;
    p.A12 = p.A / 12.0;
    p.k = k;
    p.b = b;
    return p;
}

struct V3 {
    double x, y, z;
};

__device__ __forceinline__ V3 cross(const V3& a, const V3& b)
{
    return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
// Cross product with every product rounded on its own (no FMA contraction): a x a is then exactly
// zero, as in the reference's non-fused arithmetic.  Used for S(e_i) R0.col(i), which cancels
// exactly when the foot sits at its null-force orientation (R == R0), a common resting state.
__device__ __forceinline__ V3 cross_exact(const V3& a, const V3& b)
{
    return V3{__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)),
              __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
              __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}
__device__ __forceinline__ V3 operator+(const V3& a, const V3& b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(const V3& a, const V3& b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator*(double s, const V3& a) { return V3{s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ V3 neg(const V3& a) { return V3{-a.x, -a.y, -a.z}; }

// Live inputs of one contact state (27 doubles when everything is requested).
struct State {
    V3 v, w;      // mixed twist: linear, angular
    V3 p, p0;     // link position, null-force position
    V3 e1, e2;    // R.col(0), R.col(1)
    double R02, R12, R22;  // R.col(2)   (R02, R12 only feed Rdot(2,2))
    V3 n1, n2;    // R0.col(0), R0.col(1)
};

// Results.  g is stored compactly: gd = the three equal top-left diagonal entries,
// gs = bottom-right symmetric 3x3 as {xx, xy, xz, yy, yz, zz}; every other entry of the dense
// 6x6 is a structural +0.0 (ContinuousContactModel.cpp:18,165-170).
struct Result {
    V3 force, torque;       // wrench
    V3 fhead, ftail;        // autonomous dynamics
    double gd;
    double gs[6];
    V3 y_fk, y_fb, y_tk, y_tb;  // regressor corners: (force|torque) x (spring|damper) columns
    V3 t1, t2;              // e1 x w, e2 x w = -Rdot.col(0), -Rdot.col(1): reused by the fused rollout
};

template <unsigned MASK>
__device__ __forceinline__ void eval_contact(const State& s, const Prm& q, Result& r)
{
    constexpr bool kW = (MASK & M_WRENCH) != 0;
    constexpr bool kA = (MASK & M_AUTODYN) != 0;
    constexpr bool kC = (MASK & M_CTRL) != 0;
    constexpr bool kR = (MASK & M_REGRESSOR) != 0;

    const double c = s.R22;
    const double ac = fabs(c);

    // shared by wrench / autodyn / regressor
    V3 d, sd, t1, t2, u1, u2, m1, m2, Tb;
    if constexpr (kW || kA || kR) {
        d = s.p0 - s.p;
        t1 = cross(s.e1, s.w);   // e1 x w   ( = -Rdot.col(0) )
        t2 = cross(s.e2, s.w);
        u1 = cross(s.e1, t1);    // S(e1)^2 w
        u2 = cross(s.e2, t2);
        m1 = cross_exact(s.e1, s.n1);  // S(e1) R0.col(0)
        m2 = cross_exact(s.e2, s.n2);
        r.t1 = t1;
        r.t2 = t2;
    }
    if constexpr (kW || kA) {
        sd = q.k * d - q.b * s.v;                       // k (p0 - p) - b v
        const V3 T1 = q.b * u1 + q.k * m1;
        const V3 T2 = q.b * u2 + q.k * m2;
        Tb = q.L2 * T1 + q.W2 * T2;                     // the torque bracket of :102-107
    }
    if constexpr (kW) {
        r.force = (ac * q.A) * sd;
        r.torque = (ac * q.A12) * Tb;
    }
    if constexpr (kA) {
        // Rdot(2,2) = (w x R.col(2)).z
        const double cdot = s.w.x * s.R12 - s.w.y * s.R02;
        r.fhead = q.A * (cdot * sd - (c * q.k) * s.v);
        const V3 d1 = neg(t1), d2 = neg(t2);            // Rdot.col(i) = w x e_i
        // k S(de) n + b (S(de)S(e) + S(e)S(de)) w
        const V3 Q1 = q.k * cross(d1, s.n1) + q.b * (cross(d1, t1) + cross(s.e1, cross(d1, s.w)));
        const V3 Q2 = q.k * cross(d2, s.n2) + q.b * (cross(d2, t2) + cross(s.e2, cross(d2, s.w)));
        const V3 Q = q.L2 * Q1 + q.W2 * Q2;
        r.ftail = q.A12 * (cdot * Tb + c * Q);
    }
    if constexpr (kC || kR) {
        // M = L^2 S(e1)^2 + W^2 S(e2)^2 (symmetric)
        const V3 &a = s.e1, &e = s.e2;
        const double mxx = -(q.L2 * (a.y * a.y + a.z * a.z) + q.W2 * (e.y * e.y + e.z * e.z));
        const double myy = -(q.L2 * (a.x * a.x + a.z * a.z) + q.W2 * (e.x * e.x + e.z * e.z));
        const double mzz = -(q.L2 * (a.x * a.x + a.y * a.y) + q.W2 * (e.x * e.x + e.y * e.y));
        const double mxy = q.L2 * (a.x * a.y) + q.W2 * (e.x * e.y);
        const double mxz = q.L2 * (a.x * a.z) + q.W2 * (e.x * e.z);
        const double myz = q.L2 * (a.y * a.z) + q.W2 * (e.y * e.z);
        if constexpr (kC) {
            r.gd = -(q.A * q.b) * c;
            const double sc = q.A12 * c * q.b;
            r.gs[0] = sc * mxx; r.gs[1] = sc * mxy; r.gs[2] = sc * mxz;
            r.gs[3] = sc * myy; r.gs[4] = sc * myz; r.gs[5] = sc * mzz;
        }
        if constexpr (kR) {
            const double sf = ac * q.A, st = q.A12 * ac;
            r.y_fk = sf * d;
            r.y_fb = (-sf) * s.v;
            r.y_tk = st * (q.L2 * m1 + q.W2 * m2);
            r.y_tb = st * V3{mxx * s.w.x + mxy * s.w.y + mxz * s.w.z,
                             mxy * s.w.x + myy * s.w.y + myz * s.w.z,
                             mxz * s.w.x + myz * s.w.y + mzz * s.w.z};
        }
    }
}

// Which of the 30 SoA planes can affect the requested outputs (bit i = plane i).
__host__ __device__ constexpr unsigned live_planes(unsigned mask)
{
    // v w p | R col0,col1 (9,10,12,13,15,16) | R22 (17) | p0 | R0 col0,col1 (21,22,24,25,27,28)
    unsigned all = 0;
    const unsigned vwp = 0x1FFu;                       // planes 0..8
    const unsigned e12 = (1u << 9) | (1u << 10) | (1u << 12) | (1u << 13) | (1u << 15) | (1u << 16);
    const unsigned r22 = 1u << 17;
    const unsigned r0212 = (1u << 11) | (1u << 14);
    const unsigned p0 = (1u << 18) | (1u << 19) | (1u << 20);
    const unsigned n12 = (1u << 21) | (1u << 22) | (1u << 24) | (1u << 25) | (1u << 27) | (1u << 28);
    if (mask & (M_WRENCH | M_AUTODYN | M_REGRESSOR)) all |= vwp | e12 | r22 | p0 | n12;
    if (mask & M_AUTODYN) all |= r0212;
    if (mask & M_CTRL) all |= e12 | r22;
    return all;
}

// ---- reading and writing the SoA contact state --------------------------------------------------
// 30 input planes: twist (0-5), pose p | R row-major (6-17), null pose p0 | R0 row-major (18-29);
// 4 parameter planes: length, width, spring, damper.  Lanes past the end (!on) read zeros.

// The live planes into x (x zero-initialised by the caller: dead planes stay +0.0).  This exact
// form keeps every caller's machine code unchanged; folding the LIVE test into the condition does not.
template <unsigned LIVE>
__device__ __forceinline__ void load_live_planes(const double* const (&in)[30], long long i, bool on,
                                                 double (&x)[30])
{
#pragma unroll
    for (int pl = 0; pl < 30; ++pl)
        if (LIVE & (1u << pl)) x[pl] = on ? __ldcs(in[pl] + i) : 0.0;
}

__device__ __forceinline__ State state_from_planes(const double (&x)[30])
{
    State s;
    s.v = V3{x[0], x[1], x[2]};
    s.w = V3{x[3], x[4], x[5]};
    s.p = V3{x[6], x[7], x[8]};
    s.e1 = V3{x[9], x[12], x[15]};
    s.e2 = V3{x[10], x[13], x[16]};
    s.R02 = x[11];
    s.R12 = x[14];
    s.R22 = x[17];
    s.p0 = V3{x[18], x[19], x[20]};
    s.n1 = V3{x[21], x[24], x[27]};
    s.n2 = V3{x[22], x[25], x[28]};
    return s;
}

// the uniform parameters, or (HET) this contact's parameter planes
template <bool HET>
__device__ __forceinline__ Prm load_params(const double* const (&prm)[4], const Prm& uni, long long i, bool on)
{
    Prm q = uni;
    if constexpr (HET) {
        const double l = on ? __ldcs(prm[0] + i) : 0.0, w = on ? __ldcs(prm[1] + i) : 0.0;
        const double k = on ? __ldcs(prm[2] + i) : 0.0, b = on ? __ldcs(prm[3] + i) : 0.0;
        q = make_prm(l, w, k, b);
    }
    return q;
}

// force | torque into six planes
__device__ __forceinline__ void store_wrench(double* const (&wrench)[6], long long i, const Result& r)
{
    __stcs(wrench[0] + i, r.force.x); __stcs(wrench[1] + i, r.force.y);
    __stcs(wrench[2] + i, r.force.z); __stcs(wrench[3] + i, r.torque.x);
    __stcs(wrench[4] + i, r.torque.y); __stcs(wrench[5] + i, r.torque.z);
}

// ------------------------------------------------------------------------------------------------
// Reverse mode of the wrench: gbar^T d(wrench)/d(inputs) for a cotangent gbar = (gF, gT).
// With ac = |R22|, alpha = ac A, beta = ac A/12, sd = k (p0 - p) - b v, u_i = e_i x (e_i x w),
// m_i = e_i x n_i, T_i = b u_i + k m_i, Tb = L^2 T1 + W^2 T2 and h1 = beta L^2 gT, h2 = beta W^2 gT:
//   p0: k alpha gF        p: -k alpha gF        v: -b alpha gF
//   w:  b sum_i e_i x (e_i x h_i)                         (S(e)^2 is symmetric)
//   e_i: b [h_i (e_i.w) + w (h_i.e_i) - 2 (h_i.w) e_i] + k n_i x h_i
//   n_i: k h_i x e_i
//   R22: sgn(R22) (A gF.sd + A/12 gT.Tb), sgn(+-0) = 0 (torch.abs's backward)
//   k: gF.y_fk + gT.y_tk    b: gF.y_fb + gT.y_tb          (the regressor columns)
//   L: ac W gF.sd + ac W/12 gT.Tb + 2 L beta gT.T1        W: same with L <-> W, T2.
// R02, R12 and R0's third column do not enter the wrench: their gradient is structurally zero.
// ------------------------------------------------------------------------------------------------

// gradient groups (bits of the GROUPS template argument and of vjp_live_planes)
enum : unsigned { G_TWIST = 1u, G_POSE = 2u, G_NULL = 4u, G_PARAMS = 8u };

struct VjpOut {
    V3 v, w, p, e1, e2, p0, n1, n2;
    double R22;
    double L, W, k, b;   // length, width, spring, damper
};

__device__ __forceinline__ double dot(const V3& a, const V3& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

template <unsigned G>
__device__ __forceinline__ void vjp_wrench(const State& s, const Prm& q, double length, double width,
                                           const V3& gF, const V3& gT, VjpOut& g)
{
    constexpr bool kTw = (G & G_TWIST) != 0;
    constexpr bool kPo = (G & G_POSE) != 0;
    constexpr bool kNu = (G & G_NULL) != 0;
    constexpr bool kPa = (G & G_PARAMS) != 0;

    const double c = s.R22;
    const double ac = fabs(c);
    const double alpha = ac * q.A, beta = ac * q.A12;
    const V3 h1 = (beta * q.L2) * gT, h2 = (beta * q.W2) * gT;

    if constexpr (kTw) {
        g.v = (-(q.b * alpha)) * gF;
        g.w = q.b * (cross(s.e1, cross(s.e1, h1)) + cross(s.e2, cross(s.e2, h2)));
    }
    if constexpr (kPo || kNu) {
        const V3 gp0 = (q.k * alpha) * gF;
        if constexpr (kNu) {
            g.p0 = gp0;
            g.n1 = q.k * cross(h1, s.e1);
            g.n2 = q.k * cross(h2, s.e2);
        }
        if constexpr (kPo) g.p = neg(gp0);
    }
    if constexpr (kPo) {
        const double ew1 = dot(s.e1, s.w), hw1 = dot(h1, s.w), he1 = dot(h1, s.e1);
        const double ew2 = dot(s.e2, s.w), hw2 = dot(h2, s.w), he2 = dot(h2, s.e2);
        g.e1 = q.b * (ew1 * h1 + he1 * s.w - (2.0 * hw1) * s.e1) + q.k * cross(s.n1, h1);
        g.e2 = q.b * (ew2 * h2 + he2 * s.w - (2.0 * hw2) * s.e2) + q.k * cross(s.n2, h2);
    }
    if constexpr (kPo || kPa) {
        const V3 d = s.p0 - s.p;
        const V3 sd = q.k * d - q.b * s.v;
        const V3 u1 = cross(s.e1, cross(s.e1, s.w)), u2 = cross(s.e2, cross(s.e2, s.w));
        const V3 m1 = cross_exact(s.e1, s.n1), m2 = cross_exact(s.e2, s.n2);
        const double fs = dot(gF, sd);
        const double t1 = dot(gT, q.b * u1 + q.k * m1), t2 = dot(gT, q.b * u2 + q.k * m2);
        const double ts = q.L2 * t1 + q.W2 * t2;   // gT.Tb
        if constexpr (kPo) {
            const double sg = c > 0.0 ? 1.0 : (c < 0.0 ? -1.0 : 0.0);
            g.R22 = sg * (q.A * fs + q.A12 * ts);
        }
        if constexpr (kPa) {
            g.k = alpha * dot(gF, d) + beta * (q.L2 * dot(gT, m1) + q.W2 * dot(gT, m2));
            g.b = -alpha * dot(gF, s.v) + beta * (q.L2 * dot(gT, u1) + q.W2 * dot(gT, u2));
            g.L = ac * width * (fs + ts / 12.0) + (2.0 * length * beta) * t1;
            g.W = ac * length * (fs + ts / 12.0) + (2.0 * width * beta) * t2;
        }
    }
}

// Which of the 30 SoA input planes the requested gradient groups read (bit i = plane i).  The
// cotangents (and, with per-contact parameters, the 4 parameter planes) are read by every group.
__host__ __device__ constexpr unsigned vjp_live_planes(unsigned groups)
{
    const unsigned all = live_planes(M_WRENCH);   // the 25 planes the wrench depends on
    const unsigned e12 = (1u << 9) | (1u << 10) | (1u << 12) | (1u << 13) | (1u << 15) | (1u << 16);
    const unsigned r22 = 1u << 17;
    unsigned live = 0;
    if (groups & (G_POSE | G_PARAMS)) live |= all;
    if (groups & (G_TWIST | G_NULL)) live |= e12 | r22;
    return live;
}

// The input planes of each gradient group: twist 0-5, pose 6-17, null pose 18-29.
__host__ __device__ constexpr unsigned vjp_group_planes(unsigned group)
{
    return group == G_TWIST ? 0x3Fu : group == G_POSE ? 0x3FFC0u : group == G_NULL ? 0x3FFC0000u : 0u;
}

}  // namespace blfccm
