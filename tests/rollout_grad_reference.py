"""Independent restatements of the derivative of the fused rollout's cost, for the tests of
blf_ccm_rollout_cost_vjp, and the writer of its golden fixture.

chain c = rollout*feet + foot; for t = 0..H-1: (F, T)_t = wrench(twist[t][c], pose_c(t)),
chain_cost_c += wf|F_t - Fref|^2 + wt|T_t - Tref|^2, pose_c(t+1) = one ForwardEuler step;
cost[r] = sum_foot chain_cost.  Nothing here knows the adjoint formulas of csrc/sys_kernels.cuh.

(a) torch_rollout_cost: a float64 torch restatement in matrix form (Rdot = S(w) R + rho/2
    ((R R^T)^-1 - I) R as oracle/exact_golden_sys.kin_dynamics writes it), differentiated by
    torch.autograd.
(b) dual_chain_gradient: 80-digit forward mode, dual numbers over mpmath.mpf (one tangent per
    input of the chain) run through oracle/exact_golden.closed_form and
    oracle/exact_golden_sys.euler_step.
(c) fd_chain_gradient: 80-digit central differences (h = 1e-30) of mp_chain_cost, the chain cost of
    oracle/exact_golden_sys.mp_rollout restated on mpf inputs (it rounds its inputs to double, so a
    perturbation of 1e-30 cannot pass through it); tied to mp_rollout by the CPU tests.

Gradient of one chain: a vector over its inputs, in this order -- twists (H, 6), initial pose
pos (3) + rot (9, row-major), null pose (12), params (4).

Run:  python tests/rollout_grad_reference.py   -> rewrites tests/golden/rollout_grad_golden.npz
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden", "rollout_grad_golden.npz")
REF = np.array([0.0, 0.0, 30.0, 0.1, -0.2, 0.0])
WEIGHTS = np.array([1.0, 10.0])
DIGITS = 80


# --------------------------------------------------------------------------------------------------
# inputs
# --------------------------------------------------------------------------------------------------

def _rot(rng, n, tilt=0.3):
    """n rotations (9, n) row-major: small random tilts about a random axis."""
    out = np.empty((9, n))
    for c in range(n):
        a = rng.normal(size=3)
        a *= tilt * rng.uniform(0.2, 1.0) / np.linalg.norm(a)
        th = np.linalg.norm(a)
        k = a / th
        K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        out[:, c] = (np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K).reshape(9)
    return out


def make_case(n_rollouts, feet, horizon, seed, het=False, inverted=False, at_null=False):
    """Seeded inputs of one rollout batch: dict of numpy planes.  `inverted` turns chain 1 upside
    down (R22 < 0), `at_null` puts chain 0 at its null pose."""
    rng = np.random.default_rng(seed)
    chains = n_rollouts * feet
    tw = np.concatenate([rng.normal(0, 0.05, (3, horizon * chains)), rng.normal(0, 0.3, (3, horizon * chains))])
    pos = rng.normal(0, 0.01, (3, chains))
    rot = _rot(rng, chains)
    null = np.concatenate([pos + rng.normal(0, 0.005, (3, chains)), _rot(rng, chains, 0.1)])
    if inverted and chains > 1:
        rot[:, 1] = (np.diag([1.0, -1.0, -1.0]) @ rot[:, 1].reshape(3, 3)).reshape(9)
    if at_null:
        null[:3, 0] = pos[:, 0]
        null[3:, 0] = rot[:, 0]
    uni = np.array([0.2, 0.1, 1e6, 1e4])
    prm = (uni[:, None] * rng.uniform(0.7, 1.3, (4, chains))) if het else np.repeat(uni[:, None], chains, 1)
    gcost = rng.uniform(0.5, 2.0, n_rollouts)
    return dict(n_rollouts=n_rollouts, feet=feet, horizon=horizon, twist=tw, pos=pos, rot=rot, null=null,
                params=prm, uniform=uni, het=het, grad_cost=gcost)


def chain_inputs(case, c):
    """The chain's inputs as one float vector, in the gradient order."""
    H, chains = case["horizon"], case["n_rollouts"] * case["feet"]
    tw = case["twist"].reshape(6, H, chains)[:, :, c].T.reshape(-1)
    return np.concatenate([tw, case["pos"][:, c], case["rot"][:, c], case["null"][:, c], case["params"][:, c]])


def split_groups(g, horizon):
    """A chain's gradient vector -> {twist (H, 6), pose (12), null (12), params (4)}."""
    n = 6 * horizon
    return {"twist": g[:n].reshape(horizon, 6), "pose": g[n:n + 12], "null": g[n + 12:n + 24],
            "params": g[n + 24:n + 28]}


# --------------------------------------------------------------------------------------------------
# (a) float64 torch restatement
# --------------------------------------------------------------------------------------------------

def torch_rollout_cost(n_rollouts, feet, horizon, dT, rho, tw, pos, rot, null, prm, ref, weights):
    """(n_rollouts,) cost from torch tensors tw (6, H*chains), pos (3, c), rot (9, c), null (12, c),
    prm (4, c)."""
    import torch
    from wrench_grad_reference import torch_wrench
    chains = n_rollouts * feet
    p, R = pos, rot.reshape(3, 3, chains)
    ref = torch.as_tensor(ref, dtype=tw.dtype)
    eye = torch.eye(3, dtype=tw.dtype)[:, :, None]
    mm = lambda A, B: (A[:, :, None] * B[None]).sum(1)   # batched 3x3 products over the last axis
    cost = torch.zeros(chains, dtype=tw.dtype)
    for t in range(horizon):
        x = tw[:, t * chains:(t + 1) * chains]
        wr = torch_wrench(torch.cat([x, p, R.reshape(9, chains), null]), prm)
        df, dt = wr[:3] - ref[:3, None], wr[3:] - ref[3:, None]
        cost = cost + (weights[0] * (df * df).sum(0) + weights[1] * (dt * dt).sum(0))
        v, w = x[:3], x[3:]
        z = torch.zeros_like(w[0])
        Sw = torch.stack([torch.stack([z, -w[2], w[1]]), torch.stack([w[2], z, -w[0]]),
                          torch.stack([-w[1], w[0], z])])
        Rd = mm(Sw, R)
        if rho != 0.0:
            RRt = mm(R, R.permute(1, 0, 2))
            inv = torch.linalg.inv(RRt.permute(2, 0, 1)).permute(1, 2, 0)
            Rd = Rd + mm((rho / 2) * (inv - eye), R)
        p = p + dT * v
        R = R + dT * Rd
    return cost.reshape(n_rollouts, feet).sum(1)


def torch_grads(case, dT, rho, grad_cost=None):
    """Gradients of grad_cost^T cost by torch.autograd: dict twist (6, H*c), pos, rot, null, params."""
    import torch
    names = ("twist", "pos", "rot", "null", "params")
    xs = {k: torch.tensor(case[k], dtype=torch.float64, requires_grad=True) for k in names}
    cost = torch_rollout_cost(case["n_rollouts"], case["feet"], case["horizon"], dT, rho, *(xs[k] for k in names),
                              REF, WEIGHTS)
    g = torch.as_tensor(case["grad_cost"] if grad_cost is None else grad_cost)
    gs = torch.autograd.grad(cost, [xs[k] for k in names], g)
    return {k: v.numpy() for k, v in zip(names, gs)}, cost.detach().numpy()


def chain_vector(grads, case, c):
    """Gradient dict (torch_grads / kernel layout) -> chain c's gradient vector."""
    H, chains = case["horizon"], case["n_rollouts"] * case["feet"]
    tw = grads["twist"].reshape(6, H, chains)[:, :, c].T.reshape(-1)
    return np.concatenate([tw, grads["pos"][:, c], grads["rot"][:, c], grads["null"][:, c], grads["params"][:, c]])


# --------------------------------------------------------------------------------------------------
# (b) 80-digit forward mode
# --------------------------------------------------------------------------------------------------

class Dual:
    """a + sum_j t_j eps_j over mpmath.mpf, sparse tangent; with division by a dual."""
    __slots__ = ("a", "t")

    def __init__(self, a, t=None):
        self.a = a
        self.t = t or {}

    @staticmethod
    def _lift(x):
        import mpmath as mp
        return x if isinstance(x, Dual) else Dual(mp.mpf(x))

    def __add__(self, o):
        o = Dual._lift(o)
        t = dict(self.t)
        for j, v in o.t.items():
            t[j] = t[j] + v if j in t else v
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
            t[j] = t[j] + self.a * v if j in t else self.a * v
        return Dual(self.a * o.a, t)

    __rmul__ = __mul__

    def __truediv__(self, o):
        o = Dual._lift(o)
        inv = 1 / o.a
        q = self.a * inv
        t = {j: v * inv for j, v in self.t.items()}
        for j, v in o.t.items():   # d(a/b) = da/b - a db / b^2
            d = -q * v * inv
            t[j] = t[j] + d if j in t else d
        return Dual(q, t)

    def __rtruediv__(self, o):
        return Dual._lift(o) / self

    def __abs__(self):
        s = (self.a > 0) - (self.a < 0)   # sgn(+-0) = 0
        return Dual(abs(self.a), {j: s * v for j, v in self.t.items()})


def _chain_cost(x, horizon, dT, rho, ref, weights, num, zero, one):
    """Chain cost on any number type from the chain's input vector x (gradient order), through
    closed_form and euler_step as mp_rollout runs them."""
    from oracle.exact_golden import closed_form
    from oracle.exact_golden_sys import euler_step
    n = 6 * horizon
    p = list(x[n:n + 3])
    R = [list(x[n + 3 + 3 * i:n + 6 + 3 * i]) for i in range(3)]
    p0, R0 = list(x[n + 12:n + 15]), list(x[n + 15:n + 24])
    L, W, k, b = x[n + 24:n + 28]
    acc = zero
    for t in range(horizon):
        v, w = list(x[6 * t:6 * t + 3]), list(x[6 * t + 3:6 * t + 6])
        ex = closed_form(v, w, p, [R[a][q] for a in range(3) for q in range(3)], p0, R0, L, W, k, b, zero)
        df = [ex["wrench"][q] - num(ref[q]) for q in range(3)]
        dt = [ex["wrench"][3 + q] - num(ref[3 + q]) for q in range(3)]
        acc = acc + (num(weights[0]) * sum((y * y for y in df), zero)
                     + num(weights[1]) * sum((y * y for y in dt), zero))
        p, R = euler_step(num(rho), num(dT), v, w, p, R, zero, one)
    return acc


def dual_chain_gradient(x, horizon, dT, rho, ref=REF, weights=WEIGHTS):
    """d chain_cost / d x (float64, rounded once) by forward mode at 80 digits."""
    import mpmath as mp
    with mp.workdps(DIGITS):
        num = lambda v: mp.mpf(float(v))
        xs = [Dual(num(v), {i: mp.mpf(1)}) for i, v in enumerate(x)]
        cost = _chain_cost(xs, horizon, dT, rho, ref, weights, num, Dual(mp.mpf(0)), Dual(mp.mpf(1)))
        return np.array([float(cost.t.get(i, 0)) for i in range(len(x))])


def mp_chain_cost(x, horizon, dT, rho, ref=REF, weights=WEIGHTS):
    """80-digit chain cost of the mpf input vector x (not rounded)."""
    import mpmath as mp
    with mp.workdps(DIGITS):
        num = lambda v: v if isinstance(v, mp.mpf) else mp.mpf(float(v))
        return _chain_cost([num(v) for v in x], horizon, dT, rho, ref, weights, num, mp.mpf(0), mp.mpf(1))


def fd_chain_gradient(x, horizon, dT, rho, coords, h="1e-30", ref=REF, weights=WEIGHTS):
    """Central differences of mp_chain_cost at 80 digits for the chain-input indices `coords`."""
    import mpmath as mp
    with mp.workdps(DIGITS):
        xm = [mp.mpf(float(v)) for v in x]
        hh = mp.mpf(h)
        out = []
        for i in coords:
            xp, xq = list(xm), list(xm)
            xp[i] += hh
            xq[i] -= hh
            out.append(float((mp_chain_cost(xp, horizon, dT, rho, ref, weights)
                              - mp_chain_cost(xq, horizon, dT, rho, ref, weights)) / (2 * hh)))
        return np.array(out)


# --------------------------------------------------------------------------------------------------
# errors: norm-wise per (chain, gradient group)
# --------------------------------------------------------------------------------------------------

def group_errors(got, want, horizon):
    """Chain gradient vectors -> {group: |got - want| / |want|} (absolute where |want| == 0)."""
    g, w = split_groups(np.asarray(got), horizon), split_groups(np.asarray(want), horizon)
    out = {}
    for k in g:
        den = np.linalg.norm(w[k])
        out[k] = np.linalg.norm(g[k] - w[k]) / (den if den > 0 else 1.0)
    return out


# --------------------------------------------------------------------------------------------------
# golden fixture: (b) on short horizons, (c) on sampled coordinates of long ones
# --------------------------------------------------------------------------------------------------

# (name, n_rollouts, feet, horizon, dT, rho, seed, het, inverted, at_null)
SHORT_CASES = [
    ("h1_rho0_uni", 2, 2, 1, 0.01, 0.0, 11, False, True, True),
    ("h1_rho_het", 2, 2, 1, 0.01, 0.5, 12, True, True, False),
    ("h3_rho0_het", 2, 2, 3, 0.01, 0.0, 13, True, True, True),
    ("h5_rho_uni", 2, 2, 5, 0.01, 0.5, 14, False, True, True),
    ("h6_rho_het", 2, 2, 6, 0.01, 0.02, 15, True, True, False),
    ("h6_rho0_uni", 2, 1, 6, 0.005, 0.0, 16, False, True, False),
]
LONG_CASES = [
    ("h100_rho", 1, 2, 100, 0.01, 0.02, 21, True, True, False),
    ("h100_rho0", 1, 2, 100, 0.01, 0.0, 22, False, False, True),
]
FD_SAMPLES = 8   # coordinates per long chain


def case_from_row(row):
    name, nr, feet, H, dT, rho, seed, het, inv, at_null = row
    return make_case(nr, feet, H, seed, het, inv, at_null), dT, rho


def fd_coords(horizon, seed):
    """Sampled chain-input indices: early, middle and late twists, pose, null pose, parameters."""
    rng = np.random.default_rng(seed)
    n = 6 * horizon
    tw = [int(rng.integers(0, 6)), 6 * (horizon // 2) + int(rng.integers(0, 6)), n - 6 + int(rng.integers(0, 6)),
          6 * int(rng.integers(1, horizon - 1)) + int(rng.integers(0, 6))]
    return tw + [n + int(rng.integers(0, 3)), n + 3 + int(rng.integers(0, 9)), n + 12 + int(rng.integers(0, 3)),
                 n + 24 + int(rng.integers(0, 4))][:FD_SAMPLES - 4]


def write_golden():
    data = {}
    for row in SHORT_CASES:
        case, dT, rho = case_from_row(row)
        chains = case["n_rollouts"] * case["feet"]
        data[row[0] + "/dual"] = np.stack([dual_chain_gradient(chain_inputs(case, c), case["horizon"], dT, rho)
                                           for c in range(chains)])
    for row in LONG_CASES:
        case, dT, rho = case_from_row(row)
        chains = case["n_rollouts"] * case["feet"]
        coords = [fd_coords(case["horizon"], row[6] + c) for c in range(chains)]
        data[row[0] + "/coords"] = np.array(coords)
        data[row[0] + "/fd"] = np.stack([fd_chain_gradient(chain_inputs(case, c), case["horizon"], dT, rho, coords[c])
                                         for c in range(chains)])
    np.savez_compressed(GOLDEN, **data)
    return sorted(data)


def load_golden() -> dict:
    return dict(np.load(GOLDEN))


if __name__ == "__main__":
    print(write_golden())
