"""GPU tests of the kernels behind the per-instance entry points of the C ABI, at the shapes the
C++/Python facades never use:

  ccm_single_kernel<MASK>     blf_ccm_eval_batch_host with n == 1: every mask, per-call and uniform
                              parameters, NULL state arrays for a ctrl-only mask, calls interleaved
                              across two handles (each has its own mapped result block + sequence word)
  ccm_surface_points_kernel   blf_ccm_eval_surface_points: every point of batches past one grid-stride
                              pass, the rim of the surface, NULL outputs, guard bands, m <= 0
  sys_kin_aos_kernel (mode 1) blf_sys_kinematics_integrate_host over many systems and schedules, and
  sys_axpy_steps_kernel       the joint update beside it

The C ABI is called directly so that the shape under test is the one that reaches the kernel.
References: the exact-rational golden states, exact Fractions, the C oracle, a 50-digit trajectory,
and the batched kernels that share the per-element code.  Tolerance 1e-12 norm-wise relative per
3-vector block (parity.py), scaled by the operand magnitudes where the result can cancel."""
from fractions import Fraction as F

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from bipedal_locomotion_framework_b200._capi import ERR_INVALID_ARG
from oracle.exact_golden import (exact_eval_rounded, exact_surface_point, surface_edge_points,
                                 surface_points_f64)
from oracle.exact_golden_sys import mp_trajectory
from parity import TOL, assert_ctrl_structure, assert_parity

pytestmark = pytest.mark.gpu

# out_mask bit, output name, doubles per contact
OUTPUTS = ((1, "wrench", 6), (2, "autodyn", 6), (4, "ctrl", 36), (8, "regressor", 12))
SENTINEL = -7.25e300
DEGENERATE_ROW = 8   # golden row at its null-force pose: the regressor's torque block cancels to 0
REF_PARAMS = np.array(syn.REFERENCE_TEST_PARAMS)


def ptr(a):
    return None if a is None else a.ctypes.data


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


@pytest.fixture(scope="module")
def lib(torch):
    from bipedal_locomotion_framework_b200 import _capi
    return _capi.lib()


@pytest.fixture(scope="module")
def handles(torch):
    """Two handles with the reference test's uniform parameters (each test that changes them
    restores them)."""
    from bipedal_locomotion_framework_b200.contact_models import _Handle
    hs = [_Handle(0), _Handle(0)]
    for h in hs:
        h.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    yield hs
    for h in hs:
        h.close()


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _stream(torch):
    return torch.cuda.current_stream().cuda_stream


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


# --- A. one contact state through blf_ccm_eval_batch_host (n == 1) ---------------------------------

def _single(lib, h, twist, pose, null_pose, params, mask):
    """One n == 1 call with every output buffer present and filled with SENTINEL."""
    out = {key: np.full(size, SENTINEL) for _, key, size in OUTPUTS}
    prm = None if params is None else np.ascontiguousarray(params, dtype=np.float64)
    rc = lib.blf_ccm_eval_batch_host(h.ptr, 1, ptr(twist), ptr(pose), ptr(null_pose), ptr(prm), mask,
                                     ptr(out["wrench"]), ptr(out["autodyn"]), ptr(out["ctrl"]),
                                     ptr(out["regressor"]))
    return rc, out


def _row(g, i):
    return (np.ascontiguousarray(g["twists"][i]), np.ascontiguousarray(g["poses"][i]),
            np.ascontiguousarray(g["null_poses"][i]))


def _check_against(got, ref, mask, what, rows=None):
    """Requested blocks against the exact reference; the others still hold SENTINEL.  rows: the
    golden row of each state (default: all of them, in order)."""
    rows = np.arange(ref["wrench"].shape[0]) if rows is None else np.asarray(rows)
    floor = np.where(rows == DEGENERATE_ROW, 1e-6, 1e-300)
    for bit, key, _ in OUTPUTS:
        if mask & bit:
            assert_parity(got[key], ref[key], key, floor=floor if key == "regressor" else 1e-300, what=what)
        else:
            assert np.all(got[key] == SENTINEL), f"{what}{key} written though not requested"
    if mask & 4:
        assert_ctrl_structure(got["ctrl"])


def _single_all(lib, h, g, mask, per_call_params):
    n = g["twists"].shape[0]
    got = {key: np.empty((n, size)) for _, key, size in OUTPUTS}
    for i in range(n):
        rc, out = _single(lib, h, *_row(g, i), g["params"][i] if per_call_params else None, mask)
        assert rc == 0, (i, mask, rc)
        for key in got:
            got[key][i] = out[key]
    return got


@pytest.fixture(scope="module")
def exact_uniform(golden):
    """The golden states' exact outputs at the uniform (reference test) parameters."""
    rows = [exact_eval_rounded(*_row(golden, i), REF_PARAMS) for i in range(golden["twists"].shape[0])]
    return {key: np.stack([r[key] for r in rows]) for _, key, _ in OUTPUTS}


@pytest.mark.parametrize("mask", range(1, 16))
def test_single_state_every_mask_vs_exact_golden(lib, handles, golden, mask):
    """Each golden state with its own blf_ccm_params: every requested block within TOL of the exact
    rational result; the buffers of unrequested outputs untouched."""
    got = _single_all(lib, handles[0], golden, mask, per_call_params=True)
    _check_against(got, golden, mask, f"mask {mask}, per-call params: ")


@pytest.mark.parametrize("mask", range(1, 16))
def test_single_state_uniform_params_vs_exact(lib, handles, golden, exact_uniform, mask):
    """params = NULL: the handle's uniform parameters reach the kernel."""
    got = _single_all(lib, handles[0], golden, mask, per_call_params=False)
    _check_against(got, exact_uniform, mask, f"mask {mask}, uniform params: ")


@pytest.mark.parametrize("mask", range(1, 16))
def test_single_state_vs_aos_kernel(torch, lib, handles, golden, mask):
    """ccm_single_kernel<MASK> and the AoS batch kernel both evaluate eval_contact<MASK> with the same
    parameter products (make_prm on the host here, on the device there).  The control matrix and the
    regressor come out with the same bits; the wrench and the autonomous dynamics only within the
    exact-reference bound (see the comment at the assertion)."""
    got = _single_all(lib, handles[0], golden, mask, per_call_params=True)
    n = golden["twists"].shape[0]
    dev = {key: torch.full((n, size), SENTINEL, dtype=torch.float64, device="cuda") for _, key, size in OUTPUTS}
    ins = [_dev(torch, golden[k]) for k in ("twists", "poses", "null_poses", "params")]
    rc = lib.blf_ccm_eval_batch_aos(handles[0].ptr, n, *[t.data_ptr() for t in ins], mask,
                                    *[dev[key].data_ptr() if mask & bit else None for bit, key, _ in OUTPUTS],
                                    _stream(torch))
    assert rc == 0
    aos = {key: dev[key].cpu().numpy() if mask & bit else np.full((n, size), SENTINEL) for bit, key, size in OUTPUTS}
    for bit, key in ((4, "ctrl"), (8, "regressor")):
        if mask & bit:
            diff = np.nonzero((_bits(got[key]) != _bits(aos[key])).any(axis=1))[0]
            assert diff.size == 0, f"mask {mask} {key}: states {diff[:8].tolist()} differ from the AoS kernel"
    # Not bit for bit for the wrench and the autonomous dynamics: the torque bracket
    # T = b S(e)^2 w + k S(e) n0 is a sum of two products, and nvcc contracts a different one into the
    # DFMA in each kernel.  The SASS of ccm_single_kernel<1> rounds k S(e) n0 and fuses b S(e)^2 w, where
    # k and b are kernel parameters in uniform registers; ccm_aos_kernel<1, true> rounds b S(e)^2 w and
    # fuses k S(e) n0, with k and b in per-thread registers.  Both are one rounding of the same
    # expression, so both answers are held to the exact reference instead.
    _check_against(aos, golden, mask, f"mask {mask}, AoS kernel: ")


def test_ctrl_only_needs_no_twist_or_null_pose(lib, handles, golden):
    """The control matrix reads only the pose: mask 4 with twists = NULL and null_poses = NULL
    succeeds and gives the bits of the full-input call.  A mask that reads the twist refuses NULL."""
    h = handles[1]
    for i in range(golden["twists"].shape[0]):
        tw, po, nu = _row(golden, i)
        for params in (golden["params"][i], None):
            rc, full = _single(lib, h, tw, po, nu, params, 4)
            assert rc == 0
            rc, bare = _single(lib, h, None, po, None, params, 4)
            assert rc == 0
            assert np.array_equal(_bits(bare["ctrl"]), _bits(full["ctrl"])), i
    tw, po, nu = _row(golden, 0)
    for mask in (1, 2, 8, 3, 12, 15):
        for args in ((None, po, nu), (tw, po, None)):
            rc, out = _single(lib, h, *args, golden["params"][0], mask)
            assert rc == ERR_INVALID_ARG, (mask, rc)
            assert all(np.all(v == SENTINEL) for v in out.values())
    rc, _ = _single(lib, h, tw, None, nu, golden["params"][0], 4)
    assert rc == ERR_INVALID_ARG


def test_interleaved_calls_on_two_handles(lib, handles, golden):
    """500 calls alternating between two handles, state, mask and parameters changing on every call:
    each result is its own state's golden value, never a stale read of a mapped result block."""
    n = golden["twists"].shape[0]
    het = np.arange(105, n)                 # rows with their own random parameters
    other = np.arange(0, 105)               # edge rows and rows at the reference parameters
    rng = np.random.default_rng(3)
    for c in range(500):
        i = int(rng.choice(het) if c % 2 == 0 else rng.choice(other))
        mask = 1 + (7 * c) % 15             # consecutive calls never share a mask
        h = handles[(c // 2) % 2]
        rc, out = _single(lib, h, *_row(golden, i), golden["params"][i], mask)
        assert rc == 0
        _check_against({key: v[None] for key, v in out.items()}, {key: golden[key][i:i + 1] for _, key, _ in OUTPUTS},
                       mask, f"call {c} (state {i}, mask {mask}): ", rows=[i])


# --- B. surface points ---------------------------------------------------------------------------------

GUARD = 5   # points of guard band either side of each output


def _surface_call(torch, lib, h, state, xy, force=True, torque=True):
    """blf_ccm_eval_surface_points on device xy; outputs inside guard bands of SENTINEL.
    Returns rc, force (m,3) or None, torque (m,3) or None, and whether the guards held."""
    m = xy.shape[0]
    bufs = [torch.full(((m + 2 * GUARD) * 3,), SENTINEL, dtype=torch.float64, device="cuda") if want else None
            for want in (force, torque)]
    tw, po, nu = (np.ascontiguousarray(a, dtype=np.float64) for a in state)
    xy_d = _dev(torch, xy)
    rc = lib.blf_ccm_eval_surface_points(h.ptr, ptr(tw), ptr(po), ptr(nu), m, xy_d.data_ptr(),
                                         *[b.data_ptr() + 8 * 3 * GUARD if b is not None else None for b in bufs],
                                         _stream(torch))
    outs, guards = [], True
    for b in bufs:
        if b is None:
            outs.append(None)
            continue
        a = b.cpu().numpy()
        guards = guards and bool(np.all(a[:3 * GUARD] == SENTINEL) and np.all(a[3 * (m + GUARD):] == SENTINEL))
        outs.append(a[3 * GUARD:3 * (m + GUARD)].reshape(m, 3))
    return rc, outs[0], outs[1], guards


def _check_points(got_f, got_t, state, params, xy, exact_idx, what):
    """Every point against the float64 form within TOL x operand magnitude, outside points exactly
    +0.0, and the points exact_idx against exact Fractions."""
    L, W = params[0], params[1]
    inside = ~((np.abs(xy[:, 0]) > L / 2) | (np.abs(xy[:, 1]) > W / 2))
    f, t, fmag, tmag = surface_points_f64(*state, params, xy)
    for got, ref, mag, name in ((got_f, f, fmag, "force"), (got_t, t, tmag, "torque")):
        assert np.all(np.isfinite(got)), f"{what}{name}: non-finite (unwritten) point"
        out = got[~inside]
        assert np.all(out == 0.0) and not np.signbit(out).any(), f"{what}{name}: outside point not +0.0"
        err = np.abs(got - ref).max(axis=1)
        bad = np.nonzero(inside & (err > TOL * mag))[0]
        assert bad.size == 0, f"{what}{name}: point {bad[0]} of {xy.shape[0]} err {err[bad[0]]:.3e} > TOL x {mag[bad[0]]:.3e}"
    for j in exact_idx:
        ef, et = exact_surface_point(*state, params, xy[j, 0], xy[j, 1])
        for got, ex, mag, name in ((got_f, ef, fmag, "force"), (got_t, et, tmag, "torque")):
            ref = np.array([float(c) for c in ex])
            assert np.abs(got[j] - ref).max() <= TOL * mag[j], f"{what}{name}: point {j} vs exact"


def _grid_points(device_sms):
    return 8 * device_sms * 128   # points per grid-stride pass: 8 CTAs of 128 threads per SM


def _random_points(rng, m, params):
    L, W = params[0], params[1]
    return np.stack([rng.uniform(-0.6 * L, 0.6 * L, m), rng.uniform(-0.6 * W, 0.6 * W, m)], axis=1)


@pytest.mark.parametrize("passes,extra", [(0, 1), (0, 127), (0, 128), (0, 129), (1, -1), (1, 0), (1, 1), (3, 77)],
                         ids=lambda v: str(v))
def test_surface_points_every_point(torch, lib, handles, passes, extra):
    """Batches up to three grid-stride passes past the first (P points per pass, read from the
    device): every point checked, first and last point of every pass and the rim exactly."""
    P = _grid_points(torch.cuda.get_device_properties(0).multi_processor_count)
    m = passes * P + extra
    st = syn.make_states(1, seed=61)
    state = (st["twists"][0], st["poses"][0], st["null_poses"][0])
    rng = np.random.default_rng(m)
    xy = _random_points(rng, m, REF_PARAMS)
    edge = surface_edge_points(REF_PARAMS[0], REF_PARAMS[1])
    edge_at = [0, max(0, m - len(edge))] + ([P] if m >= P + len(edge) else [])
    for s in edge_at:
        k = min(len(edge), m - s)
        xy[s:s + k] = edge[:k]
    rc, f, t, guards = _surface_call(torch, lib, handles[0], state, xy)
    assert rc == 0 and guards
    exact_idx = set()
    for s in edge_at:
        exact_idx.update(range(s, min(m, s + len(edge))))
    for p0 in range(0, m, P):
        exact_idx.update({p0, min(m, p0 + P) - 1, min(m - 1, p0 + 127), min(m - 1, p0 + 128)})
    exact_idx.update(rng.choice(m, size=min(m, 250), replace=False).tolist())
    _check_points(f, t, state, REF_PARAMS, xy, sorted(exact_idx), f"m={m}: ")


def test_surface_points_edge_states(torch, lib, handles, golden):
    """Pose at the null pose (the spring term cancels), an upside-down foot (R22 < 0), a negative
    length (every point zero), and new uniform parameters between two calls."""
    h = handles[1]
    rng = np.random.default_rng(9)
    xy = np.concatenate([surface_edge_points(REF_PARAMS[0], REF_PARAMS[1]), _random_points(rng, 400, REF_PARAMS)])
    tw, po, _ = _row(golden, 0)
    states = {"null pose": (tw * 1e-9, po, po), "R22 < 0": _row(golden, 2), "config 1": _row(golden, 0)}
    assert golden["poses"][2][11] < 0
    try:
        for name, state in states.items():
            rc, f, t, guards = _surface_call(torch, lib, h, state, xy)
            assert rc == 0 and guards
            _check_points(f, t, state, REF_PARAMS, xy, range(len(xy)), f"{name}: ")
        neg = np.array([-0.12, 0.09, 2000.0, 100.0])
        h.set_uniform_params(*neg)
        rc, f, t, guards = _surface_call(torch, lib, h, states["config 1"], xy)
        assert rc == 0 and guards
        assert np.all(f == 0.0) and np.all(t == 0.0) and not (np.signbit(f).any() or np.signbit(t).any())
        stiff = np.array([0.3, 0.15, 1e6, 1e4])
        h.set_uniform_params(*stiff)   # a later call on the same handle sees the new values
        xy2 = np.concatenate([surface_edge_points(stiff[0], stiff[1]), _random_points(rng, 400, stiff)])
        rc, f, t, guards = _surface_call(torch, lib, h, states["config 1"], xy2)
        assert rc == 0 and guards
        _check_points(f, t, states["config 1"], stiff, xy2, range(len(xy2)), "after set_uniform_params: ")
    finally:
        h.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)


def test_surface_points_null_outputs_and_arguments(torch, lib, handles):
    """force_out / torque_out = NULL leave the other output as the two-output call wrote it (past
    one pass); m = 0 launches nothing; m < 0 and a NULL xy with m > 0 are refused."""
    P = _grid_points(torch.cuda.get_device_properties(0).multi_processor_count)
    h = handles[0]
    st = syn.make_states(1, seed=62)
    state = (st["twists"][0], st["poses"][0], st["null_poses"][0])
    xy = _random_points(np.random.default_rng(4), P + 1, REF_PARAMS)
    rc, f, t, guards = _surface_call(torch, lib, h, state, xy)
    assert rc == 0 and guards
    rc, f_only, none, guards = _surface_call(torch, lib, h, state, xy, torque=False)
    assert rc == 0 and guards and none is None and np.array_equal(_bits(f_only), _bits(f))
    rc, none, t_only, guards = _surface_call(torch, lib, h, state, xy, force=False)
    assert rc == 0 and guards and none is None and np.array_equal(_bits(t_only), _bits(t))

    tw, po, nu = (np.ascontiguousarray(a) for a in state)
    xy_d = _dev(torch, xy)
    out = torch.full((8,), SENTINEL, dtype=torch.float64, device="cuda")
    before = h.launch_count
    assert lib.blf_ccm_eval_surface_points(h.ptr, ptr(tw), ptr(po), ptr(nu), 0, xy_d.data_ptr(),
                                           out.data_ptr(), out.data_ptr(), _stream(torch)) == 0
    assert h.launch_count == before
    assert lib.blf_ccm_eval_surface_points(h.ptr, ptr(tw), ptr(po), ptr(nu), -1, xy_d.data_ptr(),
                                           out.data_ptr(), out.data_ptr(), _stream(torch)) == ERR_INVALID_ARG
    assert lib.blf_ccm_eval_surface_points(h.ptr, ptr(tw), ptr(po), ptr(nu), 1, None,
                                           out.data_ptr(), out.data_ptr(), _stream(torch)) == ERR_INVALID_ARG
    assert h.launch_count == before
    assert np.all(out.cpu().numpy() == SENTINEL)


# --- C. host-array integration of many systems ------------------------------------------------------------

SCHEDULES = [(1, 0.01, 0.004), (2, 0.003, 0.003), (34, 0.003, 0.001), (200, 1e-3, 0.0)]
SYSTEM_COUNTS = [2, 127, 128, 129, 4099]
CTA = 128   # threads per CTA of sys_kin_aos_kernel


def _dts(schedule):
    n_steps, step_dT, last_dT = schedule
    return [step_dT] * (n_steps - 1) + [last_dT]


def _integrate_host(lib, h, rho, schedule, tw, pos, rot, jv=None, jp=None):
    """blf_sys_kinematics_integrate_host on copies; returns rc, positions (n,3), rotations (n,9), joints."""
    n_steps, step_dT, last_dT = schedule
    p = None if pos is None else np.array(pos, dtype=np.float64)
    r = None if rot is None else np.array(rot, dtype=np.float64)
    j = None if jp is None else np.array(jp, dtype=np.float64)
    n = 0 if tw is None else tw.shape[0]
    nj = 0 if jv is None else jv.shape[0]
    rc = lib.blf_sys_kinematics_integrate_host(h.ptr, n, rho, step_dT, last_dT, n_steps, ptr(tw), ptr(p), ptr(r),
                                               nj, ptr(jv), ptr(j))
    return rc, p, r, j


def _systems(n):
    st = syn.make_states(n, seed=83)   # includes non-orthonormal rotations
    return (np.ascontiguousarray(st["twists"]), np.ascontiguousarray(st["poses"][:, :3]),
            np.ascontiguousarray(st["poses"][:, 3:]))


def _assert_rows_within(got_p, got_r, ref_p, ref_r, idx, what):
    """Position and each rotation row (3-vector blocks) within TOL of the reference."""
    blocks = [(got_p[idx], ref_p[idx])] + [(got_r[idx, 3 * k:3 * k + 3], ref_r[idx, 3 * k:3 * k + 3]) for k in range(3)]
    for b, (got, ref) in enumerate(blocks):
        err = np.abs(got - ref).max(axis=1) / np.abs(ref).max(axis=1)
        worst = int(np.argmax(err))
        assert err[worst] <= TOL, f"{what}: system {idx[worst]} block {b} rel err {err[worst]:.3e}"


def _cta_edges(n, width):
    return sorted({i for c in range(0, n, width) for i in (c, min(n, c + width) - 1)})


@pytest.mark.parametrize("schedule", SCHEDULES, ids=lambda s: f"{s[0]}x{s[1]}+{s[2]}")
@pytest.mark.parametrize("rho", [0.0, 3.0, 20.0])
def test_integrate_host_many_systems(torch, lib, handles, oracle, rho, schedule):
    """n systems with their own twists and rotations: against the C oracle stepped on the same
    schedule, bit for bit against the SoA Euler kernel (KinematicsBatch.euler_step) stepped on the
    same dT sequence, and bit for bit against each system integrated alone."""
    from bipedal_locomotion_framework_b200.system import KinematicsBatch
    from oracle import sys_oracle as so
    h = handles[0]
    kb = KinematicsBatch(0, h)
    dts = _dts(schedule)
    for n in SYSTEM_COUNTS:
        tw, pos, rot = _systems(n)
        rc, p, r, _ = _integrate_host(lib, h, rho, schedule, tw, pos, rot)
        assert rc == 0
        what = f"n={n} rho={rho} schedule={schedule}"

        op, orr = np.ascontiguousarray(pos.T), np.ascontiguousarray(rot.T)
        for dT in dts:
            op, orr = so.euler_step_batch_soa(rho, dT, np.ascontiguousarray(tw.T), op, orr, nthreads=4)
        _assert_rows_within(p, r, op.T, orr.T, np.arange(n), what + " vs oracle")

        dp, dr = _dev(torch, pos.T), _dev(torch, rot.T)
        dtw = _dev(torch, tw.T)
        for dT in dts:
            kb.euler_step(rho, dT, dtw, dp, dr)
        soa_p, soa_r = dp.cpu().numpy().T, dr.cpu().numpy().T
        assert np.array_equal(_bits(p), _bits(soa_p)), what + ": positions differ from the SoA Euler kernel"
        assert np.array_equal(_bits(r), _bits(soa_r)), what + ": rotations differ from the SoA Euler kernel"

        for i in (range(n) if n <= 129 else _cta_edges(n, CTA)):
            rc, p1, r1, _ = _integrate_host(lib, h, rho, schedule, tw[i:i + 1], pos[i:i + 1], rot[i:i + 1])
            assert rc == 0
            assert np.array_equal(_bits(p1[0]), _bits(p[i])) and np.array_equal(_bits(r1[0]), _bits(r[i])), \
                f"{what}: system {i} differs from the same system integrated alone"


@pytest.mark.parametrize("schedule", SCHEDULES[2:], ids=lambda s: f"{s[0]}x{s[1]}+{s[2]}")
def test_integrate_host_vs_50_digit_trajectory(lib, handles, schedule):
    """32 systems of a 4 099-system call (the first and last of several CTAs among them) against the
    trajectory computed at 50 digits and rounded once."""
    n, rho = 4099, 3.0
    tw, pos, rot = _systems(n)
    rc, p, r, _ = _integrate_host(lib, handles[0], rho, schedule, tw, pos, rot)
    assert rc == 0
    rng = np.random.default_rng(17)
    idx = sorted({0, 127, 128, 255, 2047, 2048, 4095, 4096, 4097, 4098} | set(rng.choice(n, 22, replace=False).tolist()))
    ref_p, ref_r = np.empty((n, 3)), np.empty((n, 9))
    for i in idx:
        mp_p, mp_r = mp_trajectory(rho, _dts(schedule), tw[i], pos[i], rot[i])
        ref_p[i], ref_r[i] = mp_p, mp_r.reshape(9)
    _assert_rows_within(p, r, ref_p, ref_r, np.array(idx), f"schedule={schedule} vs 50 digits")


@pytest.mark.parametrize("schedule", SCHEDULES, ids=lambda s: f"{s[0]}x{s[1]}+{s[2]}")
def test_integrate_host_joint_values(lib, handles, schedule):
    """joint_pos += joint_vel * dT per step.  sys_axpy_steps_kernel compiles each step to one DFMA,
    so every value must equal fl(x + v dT) rounded once per step (emulated with Fractions); all
    values within TOL x (|x0| + |v| sum dT) of the exact sum.  Joints alone (n = 0) and beside
    systems, whose result must not change."""
    n_steps, step_dT, last_dT = schedule
    total_dT = float((n_steps - 1) * F(step_dT) + F(last_dT))
    h = handles[0]
    rng = np.random.default_rng(n_steps)
    tw, pos, rot = _systems(3)
    rc, p_alone, r_alone, _ = _integrate_host(lib, h, 2.0, schedule, tw, pos, rot)
    assert rc == 0
    for nj, with_systems in ((1, False), (255, True), (256, False), (257, True), (100_003, False)):
        x0, v = rng.uniform(-2.0, 2.0, nj), rng.uniform(-3.0, 3.0, nj)
        args = (tw, pos, rot) if with_systems else (None, None, None)
        rc, p, r, x = _integrate_host(lib, h, 2.0, schedule, *args, v, x0)
        assert rc == 0
        if with_systems:
            assert np.array_equal(_bits(p), _bits(p_alone)) and np.array_equal(_bits(r), _bits(r_alone))
        exact = x0 + v * total_dT
        assert np.all(np.abs(x - exact) <= TOL * (np.abs(x0) + np.abs(v) * total_dT)), f"nj={nj}"
        sample = range(nj) if nj <= 257 else sorted(set(_cta_edges(nj, 256)[:600]) | set(rng.choice(nj, 200).tolist()))
        for i in sample:
            xi, fv = float(x0[i]), F(float(v[i]))
            for dT in _dts(schedule):
                xi = float(F(xi) + fv * F(dT))   # one rounding per step: DFMA
            assert x[i] == xi, f"nj={nj}: value {i} is {x[i]!r}, one rounding per step gives {xi!r}"


def test_integrate_host_argument_errors(lib, handles):
    h = handles[0]
    tw, pos, rot = _systems(2)
    jv, jp = np.ones(4), np.zeros(4)
    for steps in (0, -1):
        rc, p, r, j = _integrate_host(lib, h, 1.0, (steps, 0.01, 0.01), tw, pos, rot, jv, jp)
        assert rc == ERR_INVALID_ARG and np.array_equal(p, pos) and np.array_equal(j, jp)
    for k in range(3):
        args = [tw, pos, rot]
        args[k] = None
        n = 2
        rc = lib.blf_sys_kinematics_integrate_host(h.ptr, n, 1.0, 0.01, 0.01, 3, *[ptr(a) for a in args], 0, None, None)
        assert rc == ERR_INVALID_ARG, k
    for jv_, jp_ in ((None, jp), (jv, None)):
        rc = lib.blf_sys_kinematics_integrate_host(h.ptr, 0, 1.0, 0.01, 0.01, 3, None, None, None, 4, ptr(jv_), ptr(jp_))
        assert rc == ERR_INVALID_ARG
