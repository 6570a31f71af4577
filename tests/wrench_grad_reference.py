"""Two independent restatements of the derivative of the contact wrench, for the tests of
blf_ccm_wrench_vjp_soa, and the writer of its golden fixture.

1. Exact forward mode: oracle/exact_golden.closed_form evaluated on dual numbers over Fraction, one
   tangent per input.  The wrench is polynomial in the inputs apart from |R22| (derivative sgn(R22),
   0 at R22 = +-0, the convention of torch.abs's backward), so every Jacobian entry is an exact
   rational, rounded once.  It knows nothing of the closed-form adjoints in csrc/ccm_math.cuh.
2. A float64 torch restatement in matrix form (S(e)^2 = e e^T - |e|^2 I), differentiated by
   torch.autograd.

Jacobian columns: the 25 state planes the wrench depends on (LIVE_PLANES, in plane order), then
length, width, spring, damper.

Run:  python tests/wrench_grad_reference.py   -> rewrites tests/golden/wrench_grad_exact_golden.npz
"""
from __future__ import annotations

import os
import sys
from fractions import Fraction as F

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "wrench_grad_exact_golden.npz")
DEAD_PLANES = (11, 14, 23, 26, 29)          # R02, R12, R0's third column
LIVE_PLANES = [i for i in range(30) if i not in DEAD_PLANES]
NCOLS = len(LIVE_PLANES) + 4                 # + length, width, spring, damper


class Dual:
    """a + sum_j t_j eps_j over Fraction, sparse tangent."""
    __slots__ = ("a", "t")

    def __init__(self, a, t=None):
        self.a = a
        self.t = t or {}

    @staticmethod
    def _lift(x):
        return x if isinstance(x, Dual) else Dual(F(x))

    def __add__(self, o):
        o = Dual._lift(o)
        t = dict(self.t)
        for j, v in o.t.items():
            t[j] = t.get(j, 0) + v
        return Dual(self.a + o.a, t)

    __radd__ = __add__

    def __neg__(self):
        return Dual(-self.a, {j: -v for j, v in self.t.items()})

    def __sub__(self, o):
        return self + (-Dual._lift(o))

    def __rsub__(self, o):
        return Dual._lift(o) - self

    def __mul__(self, o):
        o = Dual._lift(o)
        t = {j: v * o.a for j, v in self.t.items()}
        for j, v in o.t.items():
            t[j] = t.get(j, 0) + self.a * v
        return Dual(self.a * o.a, t)

    __rmul__ = __mul__

    def __truediv__(self, o):
        assert not isinstance(o, Dual)
        return Dual(self.a / o, {j: v / o for j, v in self.t.items()})

    def __abs__(self):
        s = (self.a > 0) - (self.a < 0)
        return Dual(abs(self.a), {j: s * v for j, v in self.t.items()})


def exact_jacobian(twist, pose, null_pose, params):
    """(6, NCOLS) Fractions: d wrench / d (live planes, length, width, spring, damper)."""
    sys.path.insert(0, ROOT)
    from oracle.exact_golden import closed_form
    x = np.concatenate([twist, pose, null_pose])
    col = {pl: c for c, pl in enumerate(LIVE_PLANES)}
    xs = [Dual(F(float(x[i])), {col[i]: F(1)} if i in col else {}) for i in range(30)]
    ps = [Dual(F(float(params[j])), {len(LIVE_PLANES) + j: F(1)}) for j in range(4)]
    out = closed_form(xs[0:3], xs[3:6], xs[6:9], xs[9:18], xs[18:21], xs[21:30], *ps, zero=Dual(F(0)))
    return [[w.t.get(c, F(0)) for c in range(NCOLS)] for w in out["wrench"]]


def write_golden():
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "ccm_exact_golden.npz")))
    n = g["twists"].shape[0]
    jac = np.empty((n, 6, NCOLS))
    for i in range(n):
        J = exact_jacobian(g["twists"][i], g["poses"][i], g["null_poses"][i], g["params"][i])
        jac[i] = [[float(v) for v in row] for row in J]
    np.savez_compressed(GOLDEN, twists=g["twists"], poses=g["poses"], null_poses=g["null_poses"],
                        params=g["params"], jacobian=jac, live_planes=np.array(LIVE_PLANES))
    return n


def load_golden() -> dict:
    return dict(np.load(GOLDEN))


# --------------------------------------------------------------------------------------------------
# float64 torch restatement
# --------------------------------------------------------------------------------------------------

def torch_wrench(planes, prm):
    """(6, n) wrench from (30, n) planes and (4, n) length, width, spring, damper (torch tensors)."""
    import torch
    v, w, p, p0 = planes[0:3], planes[3:6], planes[6:9], planes[18:21]
    R = planes[9:18].reshape(3, 3, -1)
    R0 = planes[21:30].reshape(3, 3, -1)
    L, W, k, b = prm
    eye = torch.eye(3, dtype=planes.dtype, device=planes.device)[:, :, None]

    def skew(e):
        z = torch.zeros_like(e[0])
        return torch.stack([torch.stack([z, -e[2], e[1]]), torch.stack([e[2], z, -e[0]]),
                            torch.stack([-e[1], e[0], z])])

    def sq(e):  # S(e)^2 = e e^T - |e|^2 I
        return e[:, None] * e[None, :] - (e * e).sum(0)[None, None] * eye

    mv = lambda M, x: (M * x[None]).sum(1)
    ac = torch.abs(R[2, 2])
    A = L * W
    force = ac * A * (k * (p0 - p) - b * v)
    bracket = lambda i: b * mv(sq(R[:, i]), w) + k * mv(skew(R[:, i]), R0[:, i])
    torque = ac * A / 12 * (L * L * bracket(0) + W * W * bracket(1))
    return torch.cat([force, torque])


def torch_vjp(planes, prm, grad_wrench):
    """(30, n), (4, n) numpy: gbar^T J by torch.autograd on the CPU restatement (dead planes +0.0)."""
    import torch
    x = torch.tensor(planes, dtype=torch.float64, requires_grad=True)
    q = torch.tensor(prm, dtype=torch.float64, requires_grad=True)
    gx, gq = torch.autograd.grad(torch_wrench(x, q), (x, q), torch.as_tensor(grad_wrench))
    return gx.numpy(), gq.numpy()


# --------------------------------------------------------------------------------------------------
# tolerance: every block against the larger of its norm and the magnitude of its operands
# --------------------------------------------------------------------------------------------------

# 3-vector blocks of the state gradient (v, w, p, e1, e2, p0, n1, n2) and the scalar ones
STATE_BLOCKS = [[0, 1, 2], [3, 4, 5], [6, 7, 8], [9, 12, 15], [10, 13, 16], [17], [18, 19, 20],
                [21, 24, 27], [22, 25, 28]]


def operand_magnitude(planes, prm, g):
    """(30, n), (4, n): the adjoint formulas evaluated with every factor and term in absolute value
    (a x b replaced by |a| x+ |b|) -- the scale of the rounding error of any evaluation order."""
    a = np.abs
    v, w, p, p0 = a(planes[0:3]), a(planes[3:6]), a(planes[6:9]), a(planes[18:21])
    e = [a(planes[[9, 12, 15]]), a(planes[[10, 13, 16]])]
    nn = [a(planes[[21, 24, 27]]), a(planes[[22, 25, 28]])]
    L, W, k, b = a(prm)
    gF, gT = a(g[0:3]), a(g[3:6])
    ac = a(planes[17])
    cr = lambda x, y: np.stack([x[1] * y[2] + x[2] * y[1], x[2] * y[0] + x[0] * y[2],
                                x[0] * y[1] + x[1] * y[0]])
    dot = lambda x, y: (x * y).sum(0)
    alpha, beta = ac * L * W, ac * L * W / 12
    h = [beta * L * L * gT, beta * W * W * gT]
    sd = k * (p0 + p) + b * v
    T = [b * cr(e[i], cr(e[i], w)) + k * cr(e[i], nn[i]) for i in range(2)]
    Tb = L * L * T[0] + W * W * T[1]
    fs, ts = dot(gF, sd), dot(gT, Tb)
    out = np.zeros_like(planes)
    out[0:3] = b * alpha * gF
    out[3:6] = b * (cr(e[0], cr(e[0], h[0])) + cr(e[1], cr(e[1], h[1])))
    out[6:9] = out[18:21] = k * alpha * gF
    for i, rows in enumerate(([9, 12, 15], [10, 13, 16])):
        out[rows] = b * (h[i] * dot(e[i], w) + w * dot(h[i], e[i]) + 2 * dot(h[i], w) * e[i]) + \
            k * cr(nn[i], h[i])
    out[[21, 24, 27]] = k * cr(h[0], e[0])
    out[[22, 25, 28]] = k * cr(h[1], e[1])
    out[17] = L * W * fs + L * W / 12 * ts
    t1, t2 = dot(gT, T[0]), dot(gT, T[1])
    pm = np.stack([ac * W * (fs + ts / 12) + 2 * L * beta * t1, ac * L * (fs + ts / 12) + 2 * W * beta * t2,
                   alpha * dot(gF, p0 + p) + beta * dot(gT, L * L * cr(e[0], nn[0]) + W * W * cr(e[1], nn[1])),
                   alpha * dot(gF, v) + beta * dot(gT, L * L * cr(e[0], cr(e[0], w)) + W * W * cr(e[1], cr(e[1], w)))])
    return out, pm


def vjp_errors(got_planes, got_params, ref_planes, ref_params, mag_planes, mag_params):
    """(n,) worst relative error over the state blocks and the four parameter entries; None
    arguments are skipped."""
    worst = None

    def upd(got, ref, mag):
        nonlocal worst
        num = np.abs(got - ref).max(axis=0)
        den = np.maximum(np.maximum(np.abs(ref).max(axis=0), mag.max(axis=0)), 1e-300)
        e = np.where(num == 0.0, 0.0, num / den)
        worst = e if worst is None else np.maximum(worst, e)

    if got_planes is not None:
        for blk in STATE_BLOCKS:
            upd(got_planes[blk], ref_planes[blk], mag_planes[blk])
    if got_params is not None:
        for j in range(4):
            upd(got_params[[j]], ref_params[[j]], mag_params[[j]])
    return worst


def golden_planes(gd):
    """(30, n) planes and (4, n) parameters of the golden states."""
    planes = np.ascontiguousarray(np.concatenate([gd["twists"], gd["poses"], gd["null_poses"]], axis=1).T)
    return planes, np.ascontiguousarray(gd["params"].T)


def golden_vjp(gd, g):
    """gbar^T J of the exact Jacobians for cotangents g (6, n): (30, n) with dead planes 0, (4, n)."""
    jac = gd["jacobian"]
    prod = np.einsum("nrc,rn->cn", jac, g)
    planes = np.zeros((30, jac.shape[0]))
    planes[LIVE_PLANES] = prod[:len(LIVE_PLANES)]
    return planes, prod[len(LIVE_PLANES):]


if __name__ == "__main__":
    print("wrote", write_golden(), "exact wrench Jacobians")
