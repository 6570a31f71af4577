"""Exact / high-precision evaluation of the System-component steps either side of the contact
model, and the golden-fixture writer for them (SURVEY.md section 8(f) rows 2 and 3).

TEST INFRASTRUCTURE ONLY (see sys_oracle.h).  These fixtures pin the oracle and the
CUDA path to the reference's ALGEBRA (independently of the oracle/_ref build of its sources):

* FloatingBaseSystemKinematics::dynamics + one ForwardEuler step
  (src/System/src/FloatingBaseSystemKinematics.cpp:36-73, ForwardEuler.h:45-53) is rational in the
  inputs (one 3x3 inverse), so with the double inputs taken as exact rationals the result is an
  exact rational, rounded ONCE to double.
* Multi-step rollouts (integrate -> contact model -> cost) are evaluated with mpmath at 80
  significant digits -- far below double rounding -- and rounded once at the end.
* J^T * wrench accumulation (src/System/src/FloatingBaseSystemDynamics.cpp:199-226) is polynomial:
  exact rationals.

Run:  python oracle/exact_golden_sys.py   -> rewrites tests/golden/sys_exact_golden.npz
"""
from __future__ import annotations

import os
import sys
from fractions import Fraction as F

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
sys.path.insert(0, _ROOT)

from oracle.exact_golden import closed_form  # noqa: E402


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _mm(A, B, zero):
    return [[sum((A[i][k] * B[k][j] for k in range(3)), zero) for j in range(3)] for i in range(3)]


def _inv3(M):
    """Adjugate / determinant (exact on rationals; any formula gives the same exact value)."""
    c = lambda i, j: (M[(i + 1) % 3][(j + 1) % 3] * M[(i + 2) % 3][(j + 2) % 3]
                      - M[(i + 1) % 3][(j + 2) % 3] * M[(i + 2) % 3][(j + 1) % 3])
    det = M[0][0] * c(0, 0) + M[0][1] * c(0, 1) + M[0][2] * c(0, 2)
    return [[c(j, i) / det for j in range(3)] for i in range(3)]


def kin_dynamics(rho, v, w, R, zero, one):
    """pos_dot, rot_dot on any exact number type.  R = 3x3 nested list (row-major)."""
    cols = [[R[0][j], R[1][j], R[2][j]] for j in range(3)]
    dcols = [_cross(w, c) for c in cols]                       # -(c x w) = w x c
    Rt = [[R[j][i] for j in range(3)] for i in range(3)]
    inv = _inv3(_mm(R, Rt, zero))
    M = [[(rho / 2) * (inv[i][j] - (one if i == j else zero)) for j in range(3)] for i in range(3)]
    baum = _mm(M, R, zero)
    Rd = [[dcols[j][i] + baum[i][j] for j in range(3)] for i in range(3)]
    return list(v), Rd


def euler_step(rho, dT, v, w, p, R, zero, one):
    pd, Rd = kin_dynamics(rho, v, w, R, zero, one)
    p = [p[i] + pd[i] * dT for i in range(3)]
    R = [[R[i][j] + Rd[i][j] * dT for j in range(3)] for i in range(3)]
    return p, R


def exact_euler_step(rho, dT, twist, pos, rot):
    """Fractions in, doubles (rounded once) out: (pos_dot, rot_dot, pos_new, rot_new)."""
    fr = lambda xs: [F(float(x)) for x in xs]
    v, w, p = fr(twist[:3]), fr(twist[3:]), fr(pos)
    R = [fr(np.asarray(rot).reshape(3, 3)[i]) for i in range(3)]
    rho, dT = F(float(rho)), F(float(dT))
    pd, Rd = kin_dynamics(rho, v, w, R, F(0), F(1))
    pn, Rn = euler_step(rho, dT, v, w, p, R, F(0), F(1))
    fl = lambda M: np.array([[float(x) for x in row] for row in M])
    return (np.array([float(x) for x in pd]), fl(Rd), np.array([float(x) for x in pn]), fl(Rn))


def mp_trajectory(rho, dts, twist, pos, rot, digits=50):
    """ForwardEuler steps of sizes dts (constant twist) at `digits` significant digits, rounded once
    at the end: (pos (3,), rot (3, 3)) as doubles."""
    import mpmath as mp
    with mp.workdps(digits):
        m = lambda x: mp.mpf(float(x))
        zero, one = mp.mpf(0), mp.mpf(1)
        v, w = [m(x) for x in twist[:3]], [m(x) for x in twist[3:6]]
        p = [m(x) for x in pos]
        R = [[m(x) for x in row] for row in np.asarray(rot).reshape(3, 3)]
        rho_ = m(rho)
        for dT in dts:
            p, R = euler_step(rho_, m(dT), v, w, p, R, zero, one)
        return np.array([float(x) for x in p]), np.array([[float(x) for x in row] for row in R])


def mp_rollout(n_rollouts, feet, horizon, dT, rho, twist_planes, pos, rot, null, params,
               wrench_ref, weights, digits=80):
    """80-digit rollout.  twist_planes (6, horizon*chains) time-major, pos (3,chains), rot
    (9,chains), null (12,chains), params (4,chains).  Returns doubles rounded once."""
    import mpmath as mp
    mp.mp.dps = digits
    m = lambda x: mp.mpf(float(x))
    chains = n_rollouts * feet
    n = horizon * chains
    out = {"wrench": np.empty((6, n)), "autodyn": np.empty((6, n)), "ctrl": np.empty((n, 36)),
           "pos": np.empty((3, chains)), "rot": np.empty((9, chains)),
           "chain_cost": np.empty(chains), "cost": np.empty(n_rollouts)}
    ccost = []
    zero, one = mp.mpf(0), mp.mpf(1)
    for c in range(chains):
        p = [m(pos[i, c]) for i in range(3)]
        R = [[m(rot[3 * i + j, c]) for j in range(3)] for i in range(3)]
        p0 = [m(null[i, c]) for i in range(3)]
        R0 = [m(null[3 + i, c]) for i in range(9)]
        L, W, k, b = [m(params[i, c]) for i in range(4)]
        acc = zero
        for t in range(horizon):
            i = t * chains + c
            v = [m(twist_planes[q, i]) for q in range(3)]
            w = [m(twist_planes[3 + q, i]) for q in range(3)]
            Rflat = [R[a][bq] for a in range(3) for bq in range(3)]
            ex = closed_form(v, w, p, Rflat, p0, R0, L, W, k, b, zero)
            out["wrench"][:, i] = [float(x) for x in ex["wrench"]]
            out["autodyn"][:, i] = [float(x) for x in ex["autodyn"]]
            out["ctrl"][i] = [float(x) for x in ex["ctrl"]]
            df = [ex["wrench"][q] - m(wrench_ref[q]) for q in range(3)]
            dt = [ex["wrench"][3 + q] - m(wrench_ref[3 + q]) for q in range(3)]
            acc = acc + (m(weights[0]) * sum((x * x for x in df), zero)
                         + m(weights[1]) * sum((x * x for x in dt), zero))
            p, R = euler_step(m(rho), m(dT), v, w, p, R, zero, one)
        out["pos"][:, c] = [float(x) for x in p]
        out["rot"][:, c] = [float(R[a][bq]) for a in range(3) for bq in range(3)]
        out["chain_cost"][c] = float(acc)
        ccost.append(acc)
    for r in range(n_rollouts):
        out["cost"][r] = float(sum(ccost[r * feet:(r + 1) * feet], zero))
    return out


def exact_generalized_force(cps, ncols, twists, poses, null_poses, params, jacobians, base):
    """Exact rationals: out[s] = base[s] + sum_c J_c^T wrench_c; also the exact wrenches."""
    from oracle.exact_golden import exact_eval
    n = twists.shape[0]
    ns = n // cps
    out = np.empty((ns, ncols))
    wr = np.empty((n, 6))
    J = np.asarray(jacobians).reshape(n, 6, ncols)
    for s in range(ns):
        acc = [F(float(x)) for x in base[s]]
        for c in range(cps):
            i = s * cps + c
            w = exact_eval(twists[i], poses[i], null_poses[i], params[i])["wrench"]
            wr[i] = [float(x) for x in w]
            for q in range(ncols):
                acc[q] += sum(F(float(J[i, r, q])) * w[r] for r in range(6))
        out[s] = [float(x) for x in acc]
    return out, wr


def write_golden(seed: int = 42):
    from bipedal_locomotion_framework_b200 import synthetic as syn
    rng = np.random.default_rng(seed)
    g = {}

    # ---- single Euler steps (exact rationals) ----------------------------------------------------
    n = 64
    st = syn.make_states(n, seed=seed + 20)           # includes 5 % non-orthonormal rotations
    twists = st["twists"].copy()
    pos = st["poses"][:, :3].copy()
    rot = st["poses"][:, 3:].copy()
    rot[0] = np.eye(3).reshape(9)                     # identity start (the reference test's x0)
    twists[1] = 0.0                                   # zero twist: only the Baumgarte term acts
    rot[2] = (np.eye(3) * 1.05).reshape(9)            # scaled rotation: Baumgarte pulls it back
    rot[3] = rot[3] + 0.02 * rng.uniform(-1, 1, 9)    # clearly non-orthonormal
    rho = np.where(np.arange(n) % 3 == 0, 0.0, rng.uniform(0.1, 50.0, n))
    dT = np.where(np.arange(n) % 4 == 0, 1e-4, rng.uniform(1e-4, 2e-2, n))
    pd = np.empty((n, 3)); rd = np.empty((n, 9)); pn = np.empty((n, 3)); rn = np.empty((n, 9))
    for i in range(n):
        a, b, c, d = exact_euler_step(rho[i], dT[i], twists[i], pos[i], rot[i])
        pd[i], rd[i], pn[i], rn[i] = a, b.reshape(9), c, d.reshape(9)
    g.update(step_twists=twists, step_pos=pos, step_rot=rot, step_rho=rho, step_dT=dT,
             step_pos_dot=pd, step_rot_dot=rd, step_pos_new=pn, step_rot_new=rn)

    # ---- rollouts (80 digits) ---------------------------------------------------------------------
    nr, feet, H = 5, 2, 40
    chains = nr * feet
    st = syn.make_states(chains, seed=seed + 21, heterogeneous=True)
    tw = syn.make_states(H * chains, seed=seed + 22)["twists"]
    twist_planes = np.ascontiguousarray(tw.T)                       # (6, H*chains), time-major
    pos0 = np.ascontiguousarray(st["poses"][:, :3].T)
    rot0 = np.ascontiguousarray(st["poses"][:, 3:].T)
    null = np.ascontiguousarray(st["null_poses"].T)
    params = np.ascontiguousarray(st["params"].T)
    params[:, :4] = np.array(syn.REFERENCE_TEST_PARAMS)[:, None]    # some chains: reference values
    ref = np.array([0.0, 0.0, 30.0, 0.1, -0.1, 0.0])
    wts = np.array([1.0, 25.0])
    ro_dT, ro_rho = 0.01, 2.0
    ro = mp_rollout(nr, feet, H, ro_dT, ro_rho, twist_planes, pos0, rot0, null, params, ref, wts)
    g.update(ro_shape=np.array([nr, feet, H]), ro_dT=np.array(ro_dT), ro_rho=np.array(ro_rho),
             ro_twists=twist_planes, ro_pos0=pos0, ro_rot0=rot0, ro_null=null, ro_params=params,
             ro_ref=ref, ro_weights=wts,
             **{"ro_" + k: v for k, v in ro.items()})

    # ---- J^T wrench (exact rationals) -------------------------------------------------------------
    for tag, cps, ncols, ns in (("gfa", 2, 29, 6), ("gfb", 3, 7, 5)):
        n = ns * cps
        st = syn.make_states(n, seed=seed + 23 + cps, heterogeneous=True)
        J = rng.uniform(-1.0, 1.0, (n, 6, ncols))
        base = rng.uniform(-50.0, 50.0, (ns, ncols))
        out, wr = exact_generalized_force(cps, ncols, st["twists"], st["poses"], st["null_poses"],
                                          st["params"], J, base)
        g.update({tag + "_shape": np.array([ns, cps, ncols]), tag + "_twists": st["twists"],
                  tag + "_poses": st["poses"], tag + "_null_poses": st["null_poses"],
                  tag + "_params": st["params"], tag + "_J": J, tag + "_base": base,
                  tag + "_out": out, tag + "_wrench": wr})

    os.makedirs(os.path.join(_ROOT, "tests", "golden"), exist_ok=True)
    path = os.path.join(_ROOT, "tests", "golden", "sys_exact_golden.npz")
    np.savez_compressed(path, **g)
    return path


if __name__ == "__main__":
    print("wrote", write_golden())
