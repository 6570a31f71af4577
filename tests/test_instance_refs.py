"""CPU tests that pin the references of tests/test_gpu_instance_paths.py (no GPU): the exact surface
point force against the C oracle, its float64 numpy restatement against the exact form, and the
50-digit multi-step Euler trajectory against the oracle's repeated forward_euler_step."""
import os

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from oracle.exact_golden import exact_surface_point, surface_edge_points, surface_points_f64
from oracle.exact_golden_sys import mp_trajectory
from parity import TOL

NTHREADS = max(1, (os.cpu_count() or 1))


def _points(params, n_random, seed):
    """The rim of the surface and random points in and around it."""
    L, W = abs(params[0]), abs(params[1])
    rng = np.random.default_rng(seed)
    inner = np.stack([rng.uniform(-0.7 * L, 0.7 * L, n_random), rng.uniform(-0.7 * W, 0.7 * W, n_random)], axis=1)
    return np.concatenate([surface_edge_points(L, W), inner])


def _exact(state, xy):
    f, t = zip(*(exact_surface_point(*state, x, y) for x, y in xy))
    return (np.array([[float(c) for c in v] for v in f]), np.array([[float(c) for c in v] for v in t]))


def _assert_within(got, ref, mag, what):
    err = np.abs(got - ref).max(axis=1)
    bad = err > TOL * mag
    assert not bad.any(), f"{what}: point {int(np.argmax(bad))} err {err[bad][0]:.3e} > TOL x {mag[bad][0]:.3e}"
    outside = mag == 0.0
    assert np.all(got[outside] == 0.0)


def _golden_states(golden, rows):
    return [(golden["twists"][i], golden["poses"][i], golden["null_poses"][i], golden["params"][i]) for i in rows]


ROWS = list(range(9)) + list(range(9, 201, 19))   # every edge state, a spread of the random ones


def test_exact_surface_point_matches_the_oracle(oracle, golden):
    """exact_surface_point against ccmo_get_force_at_point / ccmo_get_torque_generated_at_point on
    the golden states, on the rim of the surface and inside it, within TOL x operand magnitude."""
    for r, st in zip(ROWS, _golden_states(golden, ROWS)):
        xy = _points(st[3], 24, seed=r)
        m = oracle.ContinuousContactModel()
        assert m.initialize(dict(zip(("length", "width", "spring_coeff", "damper_coeff"), map(float, st[3]))))
        m.setState(st[0], st[1])
        m.setNullForceTransform(st[2])
        of = np.array([m.getForceAtPoint(x, y) for x, y in xy])
        ot = np.array([m.getTorqueGeneratedAtPoint(x, y) for x, y in xy])
        ef, et = _exact(st, xy)
        _, _, fmag, tmag = surface_points_f64(*st, xy)
        inside = ~((np.abs(xy[:, 0]) > st[3][0] / 2) | (np.abs(xy[:, 1]) > st[3][1] / 2))
        fmag, tmag = np.where(inside, fmag, 0.0), np.where(inside, tmag, 0.0)
        _assert_within(of, ef, fmag, f"row {r} force")
        _assert_within(ot, et, tmag, f"row {r} torque")
        assert np.all(ef[~inside] == 0.0) and np.all(et[~inside] == 0.0)


def test_surface_points_f64_matches_exact(golden):
    """The vectorised float64 form (used where m is too large for Fractions) against the exact form,
    outside points exactly +0.0 in both."""
    for r, st in zip(ROWS, _golden_states(golden, ROWS)):
        xy = _points(st[3], 40, seed=100 + r)
        f, t, fmag, tmag = surface_points_f64(*st, xy)
        ef, et = _exact(st, xy)
        inside = ~((np.abs(xy[:, 0]) > st[3][0] / 2) | (np.abs(xy[:, 1]) > st[3][1] / 2))
        _assert_within(f, ef, np.where(inside, fmag, 0.0), f"row {r} force")
        _assert_within(t, et, np.where(inside, tmag, 0.0), f"row {r} torque")
        assert not np.signbit(f[~inside]).any() and not np.signbit(t[~inside]).any()


def test_surface_edge_points_straddle_the_rim():
    L, W = syn.REFERENCE_TEST_PARAMS[:2]
    xy = surface_edge_points(L, W)
    assert xy.shape == (49, 2)
    inside = ~((np.abs(xy[:, 0]) > L / 2) | (np.abs(xy[:, 1]) > W / 2))
    assert inside.sum() == 25 and (xy[:, 0] == L / 2).sum() == 7 and (np.abs(xy[:, 0]) == np.nextafter(L / 2, 1)).sum() == 14
    assert np.signbit(xy[:, 0]).sum() == 3 * 7     # -L/2, just below it, -0.0


@pytest.mark.parametrize("n_steps,step_dT,last_dT", [(34, 0.003, 0.001), (200, 1e-3, 0.0)])
def test_mp_trajectory_matches_repeated_oracle_steps(oracle, n_steps, step_dT, last_dT):
    """mp_trajectory (50 digits, rounded once) against the C oracle's forward_euler_step repeated on
    the same schedule, within TOL per 3-vector: the reference the GPU integration tests lean on."""
    from oracle import sys_oracle as so
    st = syn.make_states(24, seed=77)
    tw, pos, rot = st["twists"], st["poses"][:, :3], st["poses"][:, 3:]
    dts = [step_dT] * (n_steps - 1) + [last_dT]
    for rho in (0.0, 3.0):
        p, r = np.ascontiguousarray(pos.T), np.ascontiguousarray(rot.T)
        for dT in dts:
            p, r = so.euler_step_batch_soa(rho, dT, np.ascontiguousarray(tw.T), p, r, nthreads=NTHREADS)
        for i in range(0, 24, 3 if rho == 0.0 else 1):
            mp_p, mp_r = mp_trajectory(rho, dts, tw[i], pos[i], rot[i])
            assert np.abs(p[:, i] - mp_p).max() <= TOL * np.abs(mp_p).max()
            for row in range(3):
                ref = mp_r[row]
                assert np.abs(r[3 * row:3 * row + 3, i] - ref).max() <= TOL * np.abs(ref).max(), (rho, i, row)
