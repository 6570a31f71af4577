"""GPU parity against THE REFERENCE BUILD: the CUDA path, called through the C ABI, compared on the
same bits with what oracle/_ref/libblf_reference.so -- the reference's own, unmodified sources compiled
against stand-in Eigen/iDynTree headers (oracle/refbuild/) -- answers.  Those answers come from
tests/reference_samples.py: the C restatement held bit for bit to that build, pinned to stored samples.
Also the drop-in check: the reference's unmodified Catch2 contact-model test, linked to the B200
facade instead of the reference's classes, passes on the GPU (only where the original project's
source tree is given, BLF_REFERENCE_ROOT).
Tolerance 1e-12 norm-wise relative per 3-vector block (north_star)."""
import os
import subprocess

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from parity import TOL, assert_ctrl_structure, assert_parity

pytestmark = pytest.mark.gpu

NTHREADS = max(1, (os.cpu_count() or 1))
FULL_R = 15
KEYS = ("wrench", "autodyn", "ctrl", "regressor")


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


@pytest.fixture(scope="module")
def ref():
    import reference_samples
    return reference_samples


@pytest.fixture(scope="module")
def ref_build():
    from oracle import ref_binding
    if not ref_binding.available():
        pytest.skip("compiles the original project's unmodified test sources: needs its tree (BLF_REFERENCE_ROOT)")
    return ref_binding


@pytest.fixture(scope="module")
def batch(torch):
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    b = ContinuousContactModelBatch(0)
    b.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    return b


def _dev(torch, a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check(got, want, what):
    worst = 0.0
    for key in KEYS:
        e, _ = assert_parity(got[key], want[key], key, what=what + " ")
        worst = max(worst, e)
    assert_ctrl_structure(got["ctrl"])
    return worst


@pytest.mark.parametrize("heterogeneous", [False, True])
@pytest.mark.parametrize("layout", ["soa", "aos", "host"])
def test_batched_evaluation_vs_reference_build(torch, batch, ref, layout, heterogeneous):
    n = 300_007  # ragged
    st = syn.make_states(n, seed=42 + 11, heterogeneous=heterogeneous)
    if not heterogeneous:
        st["uniform"] = np.array(syn.REFERENCE_TEST_PARAMS)
    want = ref.eval_batch_states(st, FULL_R, nthreads=NTHREADS)
    if layout == "soa":
        planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
        prm = _dev(torch, st["params"].T) if heterogeneous else None
        out = batch.evaluate_soa(planes, prm, FULL_R)
        got = {k: (out[k].cpu().numpy() if k == "ctrl" else out[k].cpu().numpy().T.copy()) for k in KEYS}
    elif layout == "aos":
        out = batch.evaluate_aos(_dev(torch, st["twists"]), _dev(torch, st["poses"]),
                                 _dev(torch, st["null_poses"]),
                                 _dev(torch, st["params"]) if heterogeneous else None, FULL_R)
        got = {k: out[k].cpu().numpy() for k in KEYS}
    else:
        out = batch.evaluate_host(st["twists"], st["poses"], st["null_poses"],
                                  st["params"] if heterogeneous else None, FULL_R)
        got = {k: np.asarray(out[k]) for k in KEYS}
    worst = _check(got, want, f"{layout} vs reference build")
    assert worst <= TOL


def test_golden_states_vs_reference_build(torch, batch, ref, golden):
    """The 201 edge-case states of the exact golden file (inverted foot, R22 = +-0, un-initialised
    parameters, negative length, pose == null pose), GPU against the reference build."""
    g = golden
    want = ref.eval_batch_aos(g["twists"], g["poses"], g["null_poses"], params=g["params"], mask=FULL_R)
    out = batch.evaluate_aos(_dev(torch, g["twists"]), _dev(torch, g["poses"]), _dev(torch, g["null_poses"]),
                             _dev(torch, g["params"]), FULL_R)
    got = {k: out[k].cpu().numpy() for k in KEYS}
    for key in ("wrench", "autodyn", "ctrl"):
        assert_parity(got[key], want[key], key, what="golden states ")
    floor = np.full(g["twists"].shape[0], 1e-300)
    floor[8] = 1e-6  # pose == null pose: the regressor's bottom-left block cancels to exactly 0
    assert_parity(got["regressor"], want["regressor"], "regressor", floor=floor)
    assert_ctrl_structure(got["ctrl"])


def test_reference_unmodified_test_passes_on_the_b200_facade(ref_build):
    """src/ContactModels/tests/ContinousContactModelTest.cpp, compiled UNMODIFIED against
    bipedal_locomotion_framework_b200/cpp/include and linked to libblf_contact.so (make facade in
    oracle/refbuild): Monte-Carlo integral, regressor identity, finite differences -- on the GPU."""
    exe = os.path.join(ref_build.REF_DIR, ref_build.FACADE_TEST)
    assert os.path.exists(exe), "oracle/_ref/" + ref_build.FACADE_TEST + " was not built / shipped"
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "0 failure(s)" in r.stdout and "26 assertion(s)" in r.stdout


def test_reference_unmodified_integrator_test_passes_on_the_b200_facade(ref_build):
    """src/System/tests/IntegratorTest.cpp, compiled UNMODIFIED on the facade's System classes
    (state types = the Eigen types via BLF_HAVE_EIGEN; the reference's own LinearTimeInvariantSystem
    over the facade's DynamicalSystem / ForwardEuler templates): the linear system's closed-form
    step response, and 20 000 single-step integrate() calls of FloatingBaseSystemKinematics on the
    GPU against the axis-angle closed form."""
    exe = os.path.join(ref_build.REF_DIR, ref_build.FACADE_INTEGRATOR_TEST)
    assert os.path.exists(exe), "oracle/_ref/" + ref_build.FACADE_INTEGRATOR_TEST + " was not built / shipped"
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "0 failure(s)" in r.stdout and "120001 assertion(s)" in r.stdout


def test_per_instance_facade_vs_reference_build(torch, ref):
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModel, StdImplementation
    st = syn.make_states(24, seed=3, heterogeneous=True)
    m = ContinuousContactModel(0)
    for i in range(24):
        L, W, k, b = st["params"][i]
        h = StdImplementation()
        for key, v in (("length", L), ("width", W), ("spring_coeff", k), ("damper_coeff", b)):
            h.setParameter(key, float(v))
        assert m.initialize(h)
        m.setState(st["twists"][i], st["poses"][i])
        m.setNullForceTransform(st["null_poses"][i])
        want = ref.eval_batch_aos(st["twists"][i:i + 1], st["poses"][i:i + 1], st["null_poses"][i:i + 1],
                                  params=st["params"][i:i + 1], mask=FULL_R)
        got = {"wrench": np.asarray(m.getContactWrench()).reshape(1, 6),
               "autodyn": np.asarray(m.getAutonomousDynamics()).reshape(1, 6),
               "ctrl": np.asarray(m.getControlMatrix()).reshape(1, 36),
               "regressor": np.asarray(m.getRegressor()).reshape(1, 12)}
        _check(got, want, f"facade state {i}")
        xy = np.array([[0.01, -0.02], [0.3 * L, 0.2 * W], [L, W]])
        f_ref, t_ref = ref.surface_points(st["twists"][i], st["poses"][i], st["null_poses"][i],
                                          st["params"][i], xy)
        for j, (x, y) in enumerate(xy):
            f, t = np.asarray(m.getForceAtPoint(x, y)), np.asarray(m.getTorqueGeneratedAtPoint(x, y))
            assert np.abs(f - f_ref[j]).max() <= TOL * max(np.abs(f_ref[j]).max(), 1e-300)
            assert np.abs(t - t_ref[j]).max() <= TOL * max(np.abs(t_ref[j]).max(), 1e-300)


@pytest.mark.parametrize("p,m", [(2, 6), (3, 4), (1, 1)])
def test_rls_sequences_vs_reference_build(torch, batch, ref, p, m):
    """n independent estimators on the GPU against one reference RecursiveLeastSquare object each,
    two ways.  (i) STEP parity at the north-star tolerance: at every step the GPU starts from the
    reference's own previous state, so the difference is one step's rounding; tolerance
    max(1e-12, 128 eps cond(S)) on the operand-magnitude scale (tests/test_rls.py::_assert_step --
    the reference inverts S by LU, the kernel factorises it, and P - K Y P cancels).  (ii) DRIFT:
    a second set of estimators free-runs from its own state for all 25 steps; differences compound
    with cond(S) per step, so that comparison is held to 1e-10 and is a stability check, not the
    parity claim."""
    from bipedal_locomotion_framework_b200.estimators import RecursiveLeastSquareBatch
    from test_rls import _assert_step
    rng = np.random.default_rng(10 * p + m)
    n, ns = 64, 25
    r, lam = rng.uniform(0.2, 1.5, m), 0.99
    rls = RecursiveLeastSquareBatch(batch, r, lam)
    th0, pd = rng.normal(size=(n, p)), rng.uniform(0.5, 5.0, size=(n, p))
    Y, z = rng.normal(size=(n, ns, m, p)), rng.normal(size=(n, ns, m))
    d_th = _dev(torch, th0.T)
    P0 = np.zeros((n, p, p))
    P0[:, np.arange(p), np.arange(p)] = pd
    d_P = _dev(torch, P0.reshape(n, p * p).T)
    want = [ref.rls_run(r, lam, th0[i], pd[i], Y[i], z[i]) for i in range(n)]
    worst_med = 0.0
    for s in range(ns):
        th_prev = th0 if s == 0 else np.stack([want[i][0][s - 1] for i in range(n)])
        P_prev = P0 if s == 0 else np.stack([want[i][1][s - 1] for i in range(n)])
        th_ref = np.stack([want[i][0][s] for i in range(n)])
        P_ref = np.stack([want[i][1][s] for i in range(n)])
        d_Y, d_z = _dev(torch, Y[:, s].reshape(n, m * p).T), _dev(torch, z[:, s].T)
        # (i) one step from the reference's previous state
        s_th, s_P = _dev(torch, th_prev.T), _dev(torch, P_prev.reshape(n, p * p).T)
        rls.advance(d_Y, d_z, s_th, s_P)
        med = _assert_step(s_th.cpu().numpy().T, s_P.cpu().numpy().T.reshape(n, p, p), th_ref, P_ref,
                           th_prev, P_prev, Y[:, s], z[:, s], r, lam, f"p={p} m={m} step {s}")
        worst_med = max(worst_med, med)
        # (ii) free-running
        rls.advance(d_Y, d_z, d_th, d_P)
        th = d_th.cpu().numpy().T
        P = d_P.cpu().numpy().T.reshape(n, p, p)
        for i in range(n):
            scale_th = max(np.abs(th_ref[i]).max(), np.abs(th_prev[i]).max(), 1e-2)
            scale_P = max(np.abs(P_prev[i]).max(), np.abs(P_ref[i]).max())
            assert np.abs(th[i] - th_ref[i]).max() <= 1e-10 * scale_th, (i, s)
            assert np.abs(P[i] - P_ref[i]).max() <= 1e-10 * scale_P, (i, s)
    assert worst_med <= 1e-13      # the typical estimator and step agree far below the bound


@pytest.mark.parametrize("rho", [0.0, 2.0])
def test_euler_step_vs_reference_build(torch, batch, ref, rho):
    from bipedal_locomotion_framework_b200.system import KinematicsBatch
    kb = KinematicsBatch(0, batch.handle)
    n, dT = 257, 2e-3
    st = syn.make_states(n, seed=91)
    tw = np.ascontiguousarray(st["twists"].T)
    p, r = _dev(torch, st["poses"][:, :3].T), _dev(torch, st["poses"][:, 3:].T)
    kb.euler_step(rho, dT, _dev(torch, tw), p, r)
    p, r = p.cpu().numpy().T, r.cpu().numpy().T
    for i in range(n):
        ok, p_ref, r_ref, _ = ref.kin_integrate(rho, dT, 0.0, dT, st["twists"][i], st["poses"][i, :3],
                                                st["poses"][i, 3:])
        assert ok
        assert np.abs(p[i] - p_ref).max() <= TOL * np.abs(p_ref).max()
        assert np.abs(r[i] - r_ref.reshape(9)).max() <= TOL * np.abs(r_ref).max()


@pytest.mark.parametrize("rho,het", [(0.0, False), (2.0, True)])
def test_fused_rollout_vs_reference_build(torch, batch, ref, rho, het):
    """integrate -> contact -> cost in one kernel against the reference's objects sequenced by
    ref_driver.cpp (ContinuousContactModel + ForwardEuler<FloatingBaseSystemKinematics>)."""
    from bipedal_locomotion_framework_b200.system import RolloutBatch
    from oracle import ccm_oracle
    nr, feet, H, dT = 96, 2, 40, 0.01
    chains = nr * feet
    st = syn.make_states(chains, seed=60, heterogeneous=het)
    tw = np.random.default_rng(8).uniform(-1, 1, (H, chains, 6))
    uniform = np.array(syn.REFERENCE_TEST_PARAMS)
    want = ref.rollout(tw, st["poses"], st["null_poses"], dT, rho, params=st["params"] if het else None,
                       uniform=uniform, mask=7, nthreads=NTHREADS)
    wref, wts = [0, 0, 30.0, 0, 0, 0], [1.0, 10.0]
    out = RolloutBatch(batch).run(nr, feet, H, dT, rho, _dev(torch, tw.reshape(H * chains, 6).T),
                                  _dev(torch, st["poses"][:, :3].T), _dev(torch, st["poses"][:, 3:].T),
                                  _dev(torch, st["null_poses"].T), wref, wts,
                                  param_planes=_dev(torch, st["params"].T) if het else None, mask=7,
                                  want_final=True)
    assert_parity(out["wrench"].cpu().numpy().T, want["wrench"], "wrench", what="rollout ")
    assert_parity(out["autodyn"].cpu().numpy().T, want["autodyn"], "autodyn", what="rollout ")
    assert_parity(out["ctrl"].cpu().numpy(), want["ctrl"], "ctrl", what="rollout ")
    fin = want["final_poses"]
    assert np.abs(out["final_pos"].cpu().numpy().T - fin[:, :3]).max() <= 1e-12
    assert np.abs(out["final_rot"].cpu().numpy().T - fin[:, 3:]).max() <= 1e-12
    # cost = this repository's definition applied to the reference build's wrenches
    w = want["wrench"].reshape(H, nr, feet, 6)
    d = w - np.asarray(wref)
    cost_ref = (wts[0] * (d[..., :3] ** 2).sum(-1) + wts[1] * (d[..., 3:] ** 2).sum(-1)).sum(axis=(0, 2))
    cost = out["cost"].cpu().numpy()
    assert np.allclose(cost, cost_ref, rtol=1e-12)
    assert batch.decode_best(out["best"])[1] == int(np.argmin(cost))


@pytest.mark.parametrize("cps,ncols,het", [(2, 29, False), (4, 38, True), (1, 6, False)])
def test_generalized_force_vs_reference_build(torch, batch, ref, cps, ncols, het):
    """blf_ccm_generalized_force_soa against FloatingBaseDynamicalSystem::dynamics run from the
    reference's own FloatingBaseSystemDynamics.cpp (KinDynComputations test double: identity mass
    matrix, injected Jacobians / bias forces).  Error per system against the magnitude of the summed
    terms (the sum cancels)."""
    from bipedal_locomotion_framework_b200.system import GeneralizedForceBatch
    ns = 3_001
    n = ns * cps
    st = syn.make_states(n, seed=81 + cps, heterogeneous=het)
    rng = np.random.default_rng(cps * 100 + ncols)
    J = rng.uniform(-1.0, 1.0, (n, 6, ncols))
    base = rng.uniform(-50.0, 50.0, (ns, ncols))
    want, wref = ref.generalized_force(cps, ncols, st["twists"], st["poses"], st["null_poses"], J, base,
                                       params=st["params"] if het else None,
                                       uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True, nthreads=NTHREADS)
    planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
    out, wr = GeneralizedForceBatch(batch).run(cps, ncols, planes, _dev(torch, J), _dev(torch, base),
                                               param_planes=_dev(torch, st["params"].T) if het else None,
                                               want_wrench=True)
    mag = np.abs(base) + np.einsum("scrq,scr->sq", np.abs(J.reshape(ns, cps, 6, ncols)),
                                   np.abs(wref.reshape(ns, cps, 6)))
    err = np.abs(out.cpu().numpy() - want).max(axis=1) / np.maximum(mag.max(axis=1), 1e-300)
    assert err.max() <= TOL, (int(np.argmax(err)), err.max())
    assert_parity(wr.cpu().numpy().T, wref, "wrench")
