"""Exact-arithmetic evaluation of the reference's closed form, and the golden-fixture writer.

TEST INFRASTRUCTURE ONLY (see ccm_oracle.h).  The reference's formulas
(src/ContactModels/src/ContinuousContactModel.cpp:79-171, :223-254) are polynomial in the inputs
apart from one abs() and one division by 12, so with the double inputs taken as exact rationals the
result is an exact rational; it is then rounded ONCE to the nearest double.  Any faithful
floating-point evaluation order (Eigen's, the C oracle's, the CUDA kernel's) must agree with this
to a few ulps of the block norm -- that is what pins the C oracle in the absence of reference
golden vectors (a second pin, independent of the build of the reference's own sources in oracle/_ref).

This third derivation uses cross products, not the skew-matrix products of ccm_oracle.c.

Run:  python oracle/exact_golden.py      -> rewrites tests/golden/ccm_exact_golden.npz and
                                            tests/golden/ccm_config1.json
"""
from __future__ import annotations

import json
import os
import sys
from fractions import Fraction as F

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _add(a, b):
    return [x + y for x, y in zip(a, b)]


def _scale(s, a):
    return [s * x for x in a]


def exact_eval(twist, pose, null_pose, params):
    """All four outputs of one contact state as exact Fractions.

    twist[6], pose[12], null_pose[12] (iDynTree layouts), params = (length, width, spring, damper).
    Returns dict wrench[6], autodyn[6], ctrl[36] row-major, regressor[12] row-major 6x2.
    """
    fr = lambda xs: [F(float(x)) for x in xs]
    return closed_form(fr(twist[0:3]), fr(twist[3:6]), fr(pose[0:3]), fr(pose[3:12]),
                       fr(null_pose[0:3]), fr(null_pose[3:12]), *fr(params), zero=F(0))


def closed_form(v, w, p, R, p0, R0, L, W, k, b, zero):
    """The closed form on any exact / high-precision number type (Fraction, mpmath.mpf)."""
    A = L * W
    A12 = A / 12
    c = R[8]
    absc = abs(c)
    d = [p0[i] - p[i] for i in range(3)]
    e1, e2, e3 = [R[0], R[3], R[6]], [R[1], R[4], R[7]], [R[2], R[5], R[8]]
    n1, n2 = [R0[0], R0[3], R0[6]], [R0[1], R0[4], R0[7]]
    L2, W2 = L * L, W * W

    spring_damper = [k * d[i] - b * v[i] for i in range(3)]

    def bracket(e, n):  # b S(e)S(e) w + k S(e) n
        return _add(_scale(b, _cross(e, _cross(e, w))), _scale(k, _cross(e, n)))

    Tb = _add(_scale(L2, bracket(e1, n1)), _scale(W2, bracket(e2, n2)))
    force = _scale(absc * A, spring_damper)
    torque = _scale(absc * A12, Tb)

    # Rdot = S(w) R  (column i = w x e_i)
    d1, d2 = _cross(w, e1), _cross(w, e2)
    cdot = _cross(w, e3)[2]
    head = [A * (cdot * spring_damper[i] - c * k * v[i]) for i in range(3)]

    def rate(e, de, n):  # k S(de) n + b (S(de)S(e) + S(e)S(de)) w
        return _add(_scale(k, _cross(de, n)),
                    _scale(b, _add(_cross(de, _cross(e, w)), _cross(e, _cross(de, w)))))

    Q = _add(_scale(L2, rate(e1, d1, n1)), _scale(W2, rate(e2, d2, n2)))
    tail = [A12 * (cdot * Tb[i] + c * Q[i]) for i in range(3)]

    # M = L^2 S(e1)^2 + W^2 S(e2)^2,  S(e)^2 = e e^T - |e|^2 I
    def s2(e):
        n2_ = e[0] * e[0] + e[1] * e[1] + e[2] * e[2]
        return [[e[i] * e[j] - (n2_ if i == j else zero) for j in range(3)] for i in range(3)]

    S1, S2 = s2(e1), s2(e2)
    M = [[L2 * S1[i][j] + W2 * S2[i][j] for j in range(3)] for i in range(3)]
    ctrl = [zero] * 36
    for i in range(3):
        ctrl[6 * i + i] = -A * b * c
        for j in range(3):
            ctrl[6 * (3 + i) + 3 + j] = A12 * c * b * M[i][j]

    reg = [zero] * 12
    bl = _add(_scale(L2, _cross(e1, n1)), _scale(W2, _cross(e2, n2)))
    for i in range(3):
        reg[2 * i] = absc * A * d[i]
        reg[2 * i + 1] = -absc * A * v[i]
        reg[2 * (3 + i)] = A12 * absc * bl[i]
        reg[2 * (3 + i) + 1] = A12 * absc * sum((M[i][j] * w[j] for j in range(3)), zero)

    return {"wrench": force + torque, "autodyn": head + tail, "ctrl": ctrl, "regressor": reg}


def exact_surface_point(twist, pose, null_pose, params, x, y):
    """getForceAtPoint / getTorqueGeneratedAtPoint (ContinuousContactModel.cpp:185-219) of one
    point q = (x, y, 0) as exact Fractions: (force[3], torque[3]).

    Zero outside |x| <= length/2, |y| <= width/2 (the reference tests with a strict >, so the
    boundary is inside); else f = k((p0 - p) + (R0 - R) q) - b(v + w x R q) and tau = R q x f.
    params = (length, width, spring, damper)."""
    fr = lambda xs: [F(float(v)) for v in xs]
    L, W, k, b = fr(params)
    X, Y = F(float(x)), F(float(y))
    if abs(X) > L / 2 or abs(Y) > W / 2:
        return [F(0)] * 3, [F(0)] * 3
    v, w, p, R = fr(twist[0:3]), fr(twist[3:6]), fr(pose[0:3]), fr(pose[3:12])
    p0, R0 = fr(null_pose[0:3]), fr(null_pose[3:12])
    rq = [R[3 * i] * X + R[3 * i + 1] * Y for i in range(3)]
    r0q = [R0[3 * i] * X + R0[3 * i + 1] * Y for i in range(3)]
    wrq = _cross(w, rq)
    f = [k * ((p0[i] - p[i]) + (r0q[i] - rq[i])) - b * (v[i] + wrq[i]) for i in range(3)]
    return f, _cross(rq, f)


def surface_edge_points(length, width):
    """(49, 2) points on and around the rectangle's rim: every pair of x in {+-L/2, the next double
    outside each, +-0.0, an interior value} and the same for y -- edges, corners, signed zeros."""
    hl, hw = abs(float(length)) / 2, abs(float(width)) / 2
    xs = [hl, -hl, np.nextafter(hl, np.inf), np.nextafter(-hl, -np.inf), 0.0, -0.0, 0.3 * hl]
    ys = [hw, -hw, np.nextafter(hw, np.inf), np.nextafter(-hw, -np.inf), 0.0, -0.0, -0.7 * hw]
    return np.array([[x, y] for x in xs for y in ys], dtype=np.float64)


def surface_points_f64(twist, pose, null_pose, params, xy):
    """The same closed form in plain float64 numpy for many points xy (m, 2), with the operand
    magnitudes that bound its rounding error: returns force (m, 3), torque (m, 3),
    fmag = k(|p0 - p| + |R0 q| + |R q|) + b(|v| + |w||R q|) and tmag = fmag |R q| (both (m,))."""
    twist, pose, null_pose = (np.asarray(a, dtype=np.float64) for a in (twist, pose, null_pose))
    L, W, k, b = (float(v) for v in params)
    xy = np.asarray(xy, dtype=np.float64).reshape(-1, 2)
    x, y = xy[:, 0:1], xy[:, 1:2]
    R, R0 = pose[3:12].reshape(3, 3), null_pose[3:12].reshape(3, 3)
    v, w, dp = twist[0:3], twist[3:6], null_pose[0:3] - pose[0:3]
    rq = x * R[:, 0] + y * R[:, 1]
    r0q = x * R0[:, 0] + y * R0[:, 1]
    f = k * (dp + (r0q - rq)) - b * (v + np.cross(w, rq))
    t = np.cross(rq, f)
    inside = ~((np.abs(x[:, 0]) > L / 2) | (np.abs(y[:, 0]) > W / 2))
    f[~inside] = 0.0
    t[~inside] = 0.0
    nrq = np.linalg.norm(rq, axis=1)
    fmag = (abs(k) * (np.linalg.norm(dp) + np.linalg.norm(r0q, axis=1) + nrq)
            + abs(b) * (np.linalg.norm(v) + np.linalg.norm(w) * nrq))
    return f, t, fmag, fmag * nrq


def exact_eval_rounded(twist, pose, null_pose, params):
    ex = exact_eval(twist, pose, null_pose, params)
    return {k: np.array([float(x) for x in vals]) for k, vals in ex.items()}


def exact_rollout_cost(states, rollout_len, wrench_ref, weights, params):
    """Cost of each rollout of a rollout-major batch, cost[r] = sum_e wf|F_e - Fref|^2 +
    wt|T_e - Tref|^2 over the exact wrenches of exact_eval, summed in Fraction and rounded once.

    states: dict with twists (n, 6), poses (n, 12), null_poses (n, 12); params: (n, 4) per state, or
    one (length, width, spring, damper) for all; n a multiple of rollout_len.  Repeated states are
    evaluated once."""
    tw, po, nu = (np.asarray(states[k], dtype=np.float64) for k in ("twists", "poses", "null_poses"))
    n = tw.shape[0]
    assert n % rollout_len == 0
    prm = np.asarray(params, dtype=np.float64)
    prm = np.broadcast_to(prm, (n, 4)) if prm.ndim == 1 else prm
    ref = [F(float(x)) for x in wrench_ref]
    wf, wt = F(float(weights[0])), F(float(weights[1]))
    memo = {}

    def contact_cost(i):
        key = tw[i].tobytes() + po[i].tobytes() + nu[i].tobytes() + prm[i].tobytes()
        if key not in memo:
            w = exact_eval(tw[i], po[i], nu[i], prm[i])["wrench"]
            qf = sum((w[c] - ref[c]) ** 2 for c in range(3))
            qt = sum((w[3 + c] - ref[3 + c]) ** 2 for c in range(3))
            memo[key] = wf * qf + wt * qt
        return memo[key]

    return np.array([float(sum((contact_cost(r * rollout_len + e) for e in range(rollout_len)), F(0)))
                     for r in range(n // rollout_len)])


def _edge_states():
    """Hand-picked states the random stream does not reach."""
    from bipedal_locomotion_framework_b200 import synthetic as syn

    out = []
    base = syn.reference_test_state()
    tw, po, nu = base["twists"][0], base["poses"][0], base["null_poses"][0]
    prm = np.array(syn.REFERENCE_TEST_PARAMS)
    out.append((tw, po, nu, prm))                                       # config #1
    z = np.zeros(6)
    ident = np.concatenate([np.zeros(3), np.eye(3).reshape(9)])
    out.append((z, ident, ident, prm))                                  # defaults: all zero out
    flipped = ident.copy(); flipped[3 + 8] = -1.0; flipped[3 + 4] = -1.0
    out.append((tw, flipped, nu, prm))                                  # inverted foot, R22 = -1
    edge = po.copy(); edge[3 + 8] = 0.0
    out.append((tw, edge, nu, prm))                                     # R22 == 0
    negz = po.copy(); negz[3 + 8] = -0.0
    out.append((tw, negz, nu, prm))                                     # R22 == -0.0
    out.append((tw, po, nu, np.array([0.0, 0.0, 0.0, 0.0])))            # un-initialised params
    out.append((tw, po, nu, np.array([-0.12, 0.09, 2000.0, 100.0])))    # negative length accepted
    out.append((tw * 1e3, po, nu, np.array([0.3, 0.15, 1e6, 1e4])))     # stiff, fast
    out.append((tw * 1e-9, po, po, prm))                                # at the null pose: cancellation
    return out


def exact_rls_advance(Y, z, r, lam, theta, P):
    """One RecursiveLeastSquare::advance (src/Estimators/src/RecursiveLeastSquare.cpp:120-130) in
    exact rational arithmetic.  Y m x p, z m, r m (diag of R), theta p, P p x p -> (theta, P)."""
    m, p = len(Y), len(Y[0])
    Y = [[F(float(v)) for v in row] for row in Y]
    z = [F(float(v)) for v in z]
    r = [F(float(v)) for v in r]
    lam = F(float(lam))
    th = [F(float(v)) for v in theta]
    Pm = [[F(float(v)) for v in row] for row in P]
    mul = lambda A, B: [[sum(A[i][k] * B[k][j] for k in range(len(B))) for j in range(len(B[0]))]
                        for i in range(len(A))]
    T = lambda A: [list(c) for c in zip(*A)]
    S = mul(mul(Y, Pm), T(Y))
    for i in range(m):
        S[i][i] += lam * r[i]
    # exact inverse by Gauss-Jordan on rationals
    n = m
    aug = [S[i] + [F(int(i == j)) for j in range(n)] for i in range(n)]
    for c in range(n):
        piv = next(i for i in range(c, n) if aug[i][c] != 0)
        aug[c], aug[piv] = aug[piv], aug[c]
        d = aug[c][c]
        aug[c] = [v / d for v in aug[c]]
        for i in range(n):
            if i != c and aug[i][c] != 0:
                f = aug[i][c]
                aug[i] = [a - f * b for a, b in zip(aug[i], aug[c])]
    Sinv = [row[n:] for row in aug]
    K = mul(mul(Pm, T(Y)), Sinv)
    innov = [z[i] - sum(Y[i][k] * th[k] for k in range(p)) for i in range(m)]
    th_new = [th[c] + sum(K[c][i] * innov[i] for i in range(m)) for c in range(p)]
    KYP = mul(mul(K, Y), Pm)
    P_new = [[(Pm[a][b] - KYP[a][b]) / lam for b in range(p)] for a in range(p)]
    return ([float(v) for v in th_new], [[float(v) for v in row] for row in P_new])


def write_rls_golden(n: int = 48, steps: int = 3, seed: int = 42):
    """Contact-model identification: p = 2 (spring, damper), m = 6, regressors from exact_eval of
    synthetic contact states, a few consecutive steps per estimator (exact all the way)."""
    sys.path.insert(0, _ROOT)
    from bipedal_locomotion_framework_b200 import synthetic as syn
    rng = np.random.default_rng(seed)
    st = syn.make_states(n * steps, seed=seed + 9, heterogeneous=True)
    r = np.array([0.5, 0.5, 0.5, 0.05, 0.05, 0.05])
    lam = 0.98
    Ys = np.empty((n, steps, 6, 2)); zs = np.empty((n, steps, 6))
    th = np.empty((n, steps + 1, 2)); Ps = np.empty((n, steps + 1, 2, 2))
    for e in range(n):
        true = np.array([rng.uniform(1e3, 1e5), rng.uniform(10, 1e3)])
        theta = [0.5 * true[0], 2.0 * true[1]]
        P = [[1e8, 0.0], [0.0, 1e4]]
        th[e, 0] = theta; Ps[e, 0] = P
        for t in range(steps):
            i = e * steps + t
            prm = st["params"][i].copy()
            ex = exact_eval(st["twists"][i], st["poses"][i], st["null_poses"][i], prm)
            Y = np.array([float(v) for v in ex["regressor"]]).reshape(6, 2)
            z = Y @ true + rng.normal(0, 0.1, 6)
            theta, P = exact_rls_advance(Y.tolist(), z.tolist(), r.tolist(), lam, theta, P)
            Ys[e, t] = Y; zs[e, t] = z; th[e, t + 1] = theta; Ps[e, t + 1] = P
    np.savez_compressed(os.path.join(_ROOT, "tests", "golden", "rls_exact_golden.npz"),
                        Y=Ys, z=zs, theta=th, P=Ps, r=r, lam=np.array(lam))
    return n


def write_golden(n_random: int = 96, seed: int = 42):
    sys.path.insert(0, _ROOT)
    from bipedal_locomotion_framework_b200 import synthetic as syn

    rows = list(_edge_states())
    uni = syn.make_states(n_random, seed=seed, heterogeneous=False)
    het = syn.make_states(n_random, seed=seed + 4, heterogeneous=True)
    for i in range(n_random):
        rows.append((uni["twists"][i], uni["poses"][i], uni["null_poses"][i],
                     np.array(syn.REFERENCE_TEST_PARAMS)))
    for i in range(n_random):
        rows.append((het["twists"][i], het["poses"][i], het["null_poses"][i], het["params"][i]))

    n = len(rows)
    g = {
        "twists": np.stack([r[0] for r in rows]), "poses": np.stack([r[1] for r in rows]),
        "null_poses": np.stack([r[2] for r in rows]), "params": np.stack([r[3] for r in rows]),
        "wrench": np.empty((n, 6)), "autodyn": np.empty((n, 6)), "ctrl": np.empty((n, 36)),
        "regressor": np.empty((n, 12)),
    }
    for i, r in enumerate(rows):
        ex = exact_eval_rounded(*r)
        for key in ("wrench", "autodyn", "ctrl", "regressor"):
            g[key][i] = ex[key]
    os.makedirs(os.path.join(_ROOT, "tests", "golden"), exist_ok=True)
    np.savez_compressed(os.path.join(_ROOT, "tests", "golden", "ccm_exact_golden.npz"), **g)

    # config #1 in readable form (hex floats are exact)
    ex = exact_eval_rounded(*rows[0])
    doc = {
        "what": "BASELINE.json config #1: reference test pose/params "
                "(ContinousContactModelTest.cpp:35-47), fixed twist; outputs = exact rational "
                "evaluation of ContinuousContactModel.cpp:79-171,223-254 rounded once",
        "generator": "oracle/exact_golden.py",
        "inputs": {"twist": [float(x).hex() for x in rows[0][0]],
                   "pose": [float(x).hex() for x in rows[0][1]],
                   "null_pose": [float(x).hex() for x in rows[0][2]],
                   "params_length_width_spring_damper": [float(x).hex() for x in rows[0][3]]},
        "outputs": {k: [float(x).hex() for x in v] for k, v in ex.items()},
        "outputs_decimal": {k: [repr(float(x)) for x in v] for k, v in ex.items()},
    }
    with open(os.path.join(_ROOT, "tests", "golden", "ccm_config1.json"), "w") as f:
        json.dump(doc, f, indent=1)
    return n


if __name__ == "__main__":
    print("wrote", write_golden(), "golden states")
    print("wrote", write_rls_golden(), "golden RLS estimators")
