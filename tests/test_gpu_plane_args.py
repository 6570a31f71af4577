"""GPU tests of the plane-pointer checks of every C-ABI entry point that takes arrays of SoA plane
pointers: a NULL or misaligned (4-byte offset) plane that the call reads or writes is rejected with
BLF_CCM_ERR_INVALID_ARG before anything is launched, and a NULL plane the call never touches (a
dead input plane) is accepted."""
import ctypes as C

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import _capi
from bipedal_locomotion_framework_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

N = 256          # contacts / estimators / systems' contacts per call
DEAD_STATE_PLANE = 23   # R0[1][2]: read by no output of the wrench, the regressor or the VJP


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


@pytest.fixture(scope="module")
def batch(torch):
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    b = ContinuousContactModelBatch(0)
    b.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    return b


def _host(*v):
    return (C.c_double * len(v))(*v)


class Case:
    """One entry point: named plane-pointer arrays, a call taking them, the array entry to break
    and (where the call has one) a dead entry that may be NULL."""

    def __init__(self, arrays, call, live, dead=None):
        self.arrays, self.call, self.live, self.dead = arrays, call, live, dead


def _planes(torch, keep, rows, cols, fill=None):
    t = torch.zeros((rows, cols), dtype=torch.float64, device="cuda")
    if fill is not None:
        t.copy_(torch.from_numpy(np.ascontiguousarray(fill[:rows, :cols])))
    keep.append(t)
    return [t[i].data_ptr() for i in range(rows)]


def _identity_rot(torch, keep, cols):
    t = torch.zeros((9, cols), dtype=torch.float64, device="cuda")
    t[0] = t[4] = t[8] = 1.0
    keep.append(t)
    return [t[i].data_ptr() for i in range(9)]


def _state(torch, keep):
    st = syn.make_states(N, seed=61)
    return _planes(torch, keep, 30, N, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))


def _arr(ps):
    return None if ps is None else (C.c_void_p * len(ps))(*ps)


def case_eval_soa(torch, b, keep):
    a = {"in": _state(torch, keep), "wrench": _planes(torch, keep, 6, N)}
    call = lambda a: _capi.lib().blf_ccm_eval_batch_soa(
        b.handle.ptr, N, _arr(a["in"]), None, _capi.WRENCH, _arr(a["wrench"]), None, None, None, None)
    return Case(a, call, ("in", 17), ("in", DEAD_STATE_PLANE))


def case_rollout_cost_argmin(torch, b, keep):
    a = {"in": _state(torch, keep)}
    best = torch.empty(2, dtype=torch.int64, device="cuda")
    keep.append(best)
    ref, w = _host(0, 0, 30.0, 0, 0, 0), _host(1.0, 10.0)
    keep.extend([ref, w])
    call = lambda a: _capi.lib().blf_ccm_rollout_cost_argmin_soa(
        b.handle.ptr, N // 32, 32, _arr(a["in"]), None, 0, None, None, None, ref, w, 0, None,
        best.data_ptr(), None)
    return Case(a, call, ("in", 9), ("in", DEAD_STATE_PLANE))


def case_wrench_vjp(torch, b, keep):
    gx = _planes(torch, keep, 6, N)
    a = {"in": _state(torch, keep), "grad_wrench": _planes(torch, keep, 6, N, np.ones((6, N))),
         "grad_in": gx + [None] * 24}     # twist gradients only
    call = lambda a: _capi.lib().blf_ccm_wrench_vjp_soa(
        b.handle.ptr, N, _arr(a["in"]), None, _arr(a["grad_wrench"]), _arr(a["grad_in"]), None, None)
    return Case(a, call, ("in", 17), ("in", DEAD_STATE_PLANE))


def case_rls_contacts(torch, b, keep):
    cov = np.zeros((4, N))
    cov[0] = cov[3] = 1.0
    a = {"in": _state(torch, keep), "z": _planes(torch, keep, 6, N),
         "theta": _planes(torch, keep, 2, N, np.ones((2, N))), "cov": _planes(torch, keep, 4, N, cov)}
    r = _host(*([1.0] * 6))
    keep.append(r)
    call = lambda a: _capi.lib().blf_ccm_rls_advance_contacts(
        b.handle.ptr, N, _arr(a["in"]), None, _arr(a["z"]), r, 1.0, _arr(a["theta"]), _arr(a["cov"]), None)
    return Case(a, call, ("in", 17), ("in", DEAD_STATE_PLANE))


def _case_rls_batch(torch, b, keep, r):
    p, m = 2, 6
    cov = np.zeros((p * p, N))
    cov[0] = cov[3] = 1.0
    a = {"Y": _planes(torch, keep, m * p, N, np.full((m * p, N), 0.5)), "z": _planes(torch, keep, m, N),
         "theta": _planes(torch, keep, p, N), "cov": _planes(torch, keep, p * p, N, cov)}
    r = _host(*r)
    keep.append(r)
    call = lambda a: _capi.lib().blf_rls_advance_batch(
        b.handle.ptr, N, p, m, _arr(a["Y"]), _arr(a["z"]), r, 1.0, _arr(a["theta"]), _arr(a["cov"]), None)
    return Case(a, call, ("Y", 7))


def case_rls_batch(torch, b, keep):
    return _case_rls_batch(torch, b, keep, [1.0] * 6)


def case_rls_batch_general(torch, b, keep):
    # a zero measurement variance leaves the fast path: the pivoted-LU kernel
    return _case_rls_batch(torch, b, keep, [1.0] * 5 + [0.0])


def case_generalized_force(torch, b, keep):
    cps, ncols = 4, 6
    jac = torch.zeros((N, 6, ncols), dtype=torch.float64, device="cuda")
    out = torch.zeros((N // cps, ncols), dtype=torch.float64, device="cuda")
    keep.extend([jac, out])
    a = {"in": _state(torch, keep), "wrench": _planes(torch, keep, 6, N)}
    call = lambda a: _capi.lib().blf_ccm_generalized_force_soa(
        b.handle.ptr, N // cps, cps, ncols, _arr(a["in"]), None, jac.data_ptr(), None, out.data_ptr(),
        _arr(a["wrench"]), None)
    return Case(a, call, ("in", 17), ("in", DEAD_STATE_PLANE))


def case_rollout_integrate_cost(torch, b, keep):
    n_rollouts, feet, horizon = 64, 2, 8
    chains = n_rollouts * feet
    st = syn.make_states(chains, seed=62)
    nul = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])[18:30]
    best = torch.empty(2, dtype=torch.int64, device="cuda")
    keep.append(best)
    ref, w = _host(0, 0, 30.0, 0, 0, 0), _host(1.0, 10.0)
    keep.extend([ref, w])
    a = {"twist": _planes(torch, keep, 6, horizon * chains), "pos": _planes(torch, keep, 3, chains),
         "rot": _identity_rot(torch, keep, chains), "null": _planes(torch, keep, 12, chains, nul)}
    call = lambda a: _capi.lib().blf_ccm_rollout_integrate_cost(
        b.handle.ptr, n_rollouts, feet, horizon, 0.01, 0.0, _arr(a["twist"]), _arr(a["pos"]),
        _arr(a["rot"]), _arr(a["null"]), None, 0, None, None, None, None, None, ref, w, 0, None,
        best.data_ptr(), None)
    return Case(a, call, ("twist", 2), ("null", 5))     # R0's third column is never read


def case_kinematics_euler(torch, b, keep):
    a = {"twist": _planes(torch, keep, 6, N), "pos": _planes(torch, keep, 3, N),
         "rot": _identity_rot(torch, keep, N)}
    call = lambda a: _capi.lib().blf_sys_kinematics_euler_step_soa(
        b.handle.ptr, N, 0.0, 0.01, _arr(a["twist"]), _arr(a["pos"]), _arr(a["rot"]), None)
    return Case(a, call, ("rot", 4))


CASES = {f.__name__[5:]: f for f in (
    case_eval_soa, case_rollout_cost_argmin, case_wrench_vjp, case_rls_contacts, case_rls_batch,
    case_rls_batch_general, case_generalized_force, case_rollout_integrate_cost, case_kinematics_euler)}


# entry points whose planes are all read or written
NO_DEAD = {"rls_batch", "rls_batch_general", "kinematics_euler"}


@pytest.mark.parametrize("entry,kind", [(e, k) for e in sorted(CASES) for k in ("null", "misaligned", "dead_null")
                                        if not (k == "dead_null" and e in NO_DEAD)])
def test_plane_pointer_checks(torch, batch, entry, kind):
    keep = []
    case = CASES[entry](torch, batch, keep)
    arrays = {k: list(v) for k, v in case.arrays.items()}
    name, i = case.dead if kind == "dead_null" else case.live
    assert arrays[name][i] is not None
    arrays[name][i] = arrays[name][i] + 4 if kind == "misaligned" else None
    before = batch.handle.launch_count
    rc = case.call(arrays)
    if kind == "dead_null":
        assert rc == _capi.OK, _capi.lib().blf_ccm_last_error().decode()
        assert batch.handle.launch_count > before
    else:
        assert rc == _capi.ERR_INVALID_ARG, f"{entry}: {name}[{i}] {kind} gave {rc}"
        assert batch.handle.launch_count == before
    torch.cuda.synchronize()
