"""CPU tests that PIN THE ORACLE AGAINST THE REFERENCE'S OWN SOURCES (no GPU).

oracle/_ref/libblf_reference.so is the reference's unmodified .cpp files compiled from the original
project's tree named by BLF_REFERENCE_ROOT against stand-in Eigen/iDynTree headers (oracle/refbuild/).  Here:
  * the reference's own Catch2 tests (ContinousContactModelTest.cpp, IntegratorTest.cpp,
    ParametersHandlerTest.cpp), compiled unmodified, pass on that build -- which validates the
    stand-in headers through the reference's own properties (Monte-Carlo integral, regressor
    identity, finite differences, closed-form integration);
  * the C restatement (oracle/*.c) is compared with the reference build on seeded states; the two
    follow the same expression structure and agree BIT FOR BIT, which the tests require;
  * the reference build is compared with the exact-rational golden vectors;
  * the reference's error / lazy-cache behaviour is observed and pinned.
The tests skip (not fail) where neither that tree nor a prebuilt oracle/_ref exists.
"""
import json
import os

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from parity import assert_ctrl_structure, assert_parity

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASK_ALL = 15
DEGENERATE_ROW = 8


@pytest.fixture(scope="module")
def ref():
    from oracle import ref_binding
    if not ref_binding.available():
        pytest.skip("oracle/_ref is not built and BLF_REFERENCE_ROOT names no reference tree to build it from")
    ref_binding.build()  # refresh when the reference tree is here (make is incremental)
    return ref_binding


@pytest.fixture(scope="module")
def sys_oracle():
    from oracle import ccm_oracle, sys_oracle
    ccm_oracle.build()
    return sys_oracle


# --- the reference's own tests, unmodified, on the reference's own sources -------------------------

@pytest.mark.parametrize("exe", ["ContinuousContactModelReferenceTests", "IntegratorReferenceTests",
                                 "ParametersHandlerReferenceTests"])
def test_reference_own_tests_pass(ref, exe):
    r = ref.run_reference_test(exe)
    assert r.returncode == 0, r.stdout[-2000:]
    assert "0 failure(s)" in r.stdout


def test_reference_parameters_handler_test_passes_on_the_facade_handler(ref):
    """src/ParametersHandler/tests/ParametersHandlerTest.cpp, unmodified, on the facade's
    StdImplementation: typed getters, the VectorResizeMode contract, groups through the inherited
    shared_ptr typedefs, set-from-object, isEmpty / clear."""
    exe = os.path.join(ref.REF_DIR, ref.FACADE_HANDLER_TEST)
    if not os.path.exists(exe):
        pytest.skip("facade test binaries are built only where the product libraries exist")
    r = ref.run_reference_test(ref.FACADE_HANDLER_TEST)
    assert r.returncode == 0, r.stdout[-2000:]
    assert "20 assertion(s), 0 failure(s)" in r.stdout


def test_reference_lti_system_integrates_under_the_facade_templates(ref):
    """The reference's IntegratorTest.cpp built on the FACADE's System templates: its first section
    (the reference's own LinearTimeInvariantSystem under the facade's DynamicalSystem / ForwardEuler,
    20 000 steps against the closed-form step response) is host-only and must pass here; the second
    section needs the GPU and must fail loudly -- not fall back -- without one."""
    import torch
    exe = os.path.join(ref.REF_DIR, ref.FACADE_INTEGRATOR_TEST)
    if not os.path.exists(exe):
        pytest.skip("facade test binaries are built only where the product libraries exist")
    r = ref.run_reference_test(ref.FACADE_INTEGRATOR_TEST)
    if torch.cuda.is_available():
        assert r.returncode == 0 and "0 failure(s)" in r.stdout
        return
    assert r.returncode != 0
    assert r.stdout.count("FAILED") == 1
    assert "[section: Floating base System Kinematics]" in r.stdout
    assert "there is no CPU evaluation path" in r.stdout
    assert "40005 assertion(s), 1 failure(s)" in r.stdout   # 40 004 passed: the whole linear-system section


# --- contact model: oracle == reference build ------------------------------------------------------

@pytest.mark.parametrize("heterogeneous", [False, True])
def test_oracle_bit_identical_to_reference_build(oracle, ref, heterogeneous):
    st = syn.make_states(100_000, seed=42 + 7, heterogeneous=heterogeneous)
    a = oracle.eval_batch_states(st, MASK_ALL, nthreads=4)
    b = ref.eval_batch_states(st, MASK_ALL, nthreads=4)
    for key in ("wrench", "autodyn", "ctrl", "regressor"):
        assert np.array_equal(a[key], b[key]), f"{key}: the C restatement deviates from the reference build"
        # the sign of zero too (structural +0.0 of the control matrix)
        assert np.array_equal(np.signbit(a[key]), np.signbit(b[key]))
    assert_ctrl_structure(b["ctrl"])


def test_reference_build_matches_exact_golden(ref, golden):
    g = golden
    r = ref.eval_batch_aos(g["twists"], g["poses"], g["null_poses"], params=g["params"], mask=MASK_ALL)
    for key in ("wrench", "autodyn", "ctrl"):
        assert_parity(r[key], g[key], key, tol=1e-13, what="reference build vs exact ")
    floor = np.full(g["twists"].shape[0], 1e-300)
    floor[DEGENERATE_ROW] = 1e-6
    assert_parity(r["regressor"], g["regressor"], "regressor", tol=1e-13, floor=floor)
    assert_ctrl_structure(r["ctrl"])


def test_reference_build_config1(ref):
    """configs[0]: the reference test's pose and parameters; the committed hex-float fixture and the
    survey's independent numpy spot values."""
    with open(os.path.join(ROOT, "tests", "golden", "ccm_config1.json")) as f:
        doc = json.load(f)
    h = lambda xs: np.array([float.fromhex(x) for x in xs])
    inp, out = doc["inputs"], doc["outputs"]
    r = ref.eval_batch_aos(h(inp["twist"])[None], h(inp["pose"])[None], h(inp["null_pose"])[None],
                           uniform=h(inp["params_length_width_spring_damper"]), mask=MASK_ALL)
    for key in ("wrench", "autodyn", "ctrl", "regressor"):
        assert_parity(r[key], h(out[key])[None], key, tol=1e-13)
    np.testing.assert_allclose(r["wrench"][0],
                               [0.10465864055508661, 0.5232932027754331, -0.31397592166525984,
                                0.00225286497312795, -0.00562724183603653, -0.00591291217506123],
                               rtol=1e-12)
    assert r["ctrl"][0, 0] == pytest.approx(-1.0465864055508662, rel=1e-14)


def test_surface_points_oracle_vs_reference_build(oracle, ref):
    st = syn.reference_test_state()
    L, W, k, b = syn.REFERENCE_TEST_PARAMS
    rng = np.random.default_rng(42)
    xy = np.stack([rng.uniform(-0.6 * L, 0.6 * L, 500), rng.uniform(-0.6 * W, 0.6 * W, 500)], axis=1)
    xy[:4] = [[L / 2, W / 2], [-L / 2, -W / 2], [np.nextafter(L / 2, 1), 0.0], [0.0, 0.0]]
    f_ref, t_ref = ref.surface_points(st["twists"][0], st["poses"][0], st["null_poses"][0],
                                      (L, W, k, b), xy)
    m = oracle.ContinuousContactModel()
    assert m.initialize({"length": L, "width": W, "spring_coeff": k, "damper_coeff": b})
    m.setState(st["twists"][0], st["poses"][0])
    m.setNullForceTransform(st["null_poses"][0])
    outside = 0
    for i, (x, y) in enumerate(xy):
        assert np.array_equal(m.getForceAtPoint(x, y), f_ref[i])
        assert np.array_equal(m.getTorqueGeneratedAtPoint(x, y), t_ref[i])
        outside += int(abs(x) > L / 2 or abs(y) > W / 2)
        if abs(x) > L / 2 or abs(y) > W / 2:
            assert not f_ref[i].any() and not t_ref[i].any()
    assert outside > 10 and f_ref[0].any()  # the rectangle's border belongs to the surface


def test_reference_lazy_cache_and_initialize_behaviour(oracle, ref):
    """ContactModel.cpp:12-92 / ContinuousContactModel.cpp:24-65,256-274 observed on the reference
    build, and the oracle object behaving the same."""
    st = syn.reference_test_state()
    par = syn.REFERENCE_TEST_PARAMS
    first, stale, fresh = ref.stale_cache_probe(st["twists"][0], st["poses"][0], st["null_poses"][0],
                                                par, 3500.0)
    assert np.array_equal(first, stale)          # writing springCoeff() does not invalidate
    assert not np.array_equal(first, fresh)      # the next setState does
    m = oracle.ContinuousContactModel()
    L, W, k, b = par
    assert m.initialize({"length": L, "width": W, "spring_coeff": k, "damper_coeff": b})
    m.setState(st["twists"][0], st["poses"][0])
    m.setNullForceTransform(st["null_poses"][0])
    assert np.array_equal(m.getContactWrench(), first)
    m.springCoeff = 3500.0
    assert np.array_equal(m.getContactWrench(), stale)
    m.setState(st["twists"][0], st["poses"][0])
    assert np.array_equal(m.getContactWrench(), fresh)
    # initialize(): expired handler, each key missing, wrong type -> false; all four doubles -> true
    assert [ref.initialize_probe(w) for w in range(0, 6)] == [False] * 6
    assert ref.initialize_probe(6) is True


# --- RecursiveLeastSquare --------------------------------------------------------------------------

@pytest.mark.parametrize("p,m", [(1, 1), (2, 2), (2, 6), (3, 6), (4, 3)])
def test_rls_oracle_vs_reference_build(oracle, ref, p, m):
    rng = np.random.default_rng(100 * p + m)
    ns = 60
    Y, z = rng.normal(size=(ns, m, p)), rng.normal(size=(ns, m))
    r, lam = rng.uniform(0.1, 2.0, size=m), 0.98
    th0, pd = rng.normal(size=p), rng.uniform(0.5, 5.0, size=p)
    th_ref, P_ref = ref.rls_run(r, lam, th0, pd, Y, z)
    th, P = th0[None].copy(), np.diag(pd)[None].copy()
    for s in range(ns):
        th, P = oracle.rls_advance_batch(Y[s][None], z[s][None], r, lam, th, P)
        assert np.array_equal(th[0], th_ref[s]) and np.array_equal(P[0], P_ref[s]), f"step {s}"


def test_rls_reference_build_recovers_parameters(ref):
    """The property of src/Estimators/tests/RecursiveLeastSquareTest.cpp (which itself needs YARP):
    y = [x, x^2; sin x, cos x] theta + noise, 10 000 steps, theta within 0.1 % of (43.2, 12.2)."""
    rng = np.random.default_rng(42)
    theta_true = np.array([43.2, 12.2])
    ns = 10_000
    x = np.arange(ns) * 0.01
    Y = np.stack([np.stack([x, x * x], 1), np.stack([np.sin(x), np.cos(x)], 1)], 1)
    z = Y @ theta_true + rng.normal(0.0, 0.5, size=(ns, 2))
    th, _ = ref.rls_run([1.0, 1.0], 1.0, [0.0, 0.0], [10.0, 10.0], Y, z)
    assert np.all(np.abs(th[-1] - theta_true) / theta_true < 1e-3)


# --- FloatingBaseSystemKinematics + ForwardEuler ---------------------------------------------------

def _rand_rot(rng, perturb):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    w, x, y, z = q
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                  [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                  [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    return R + (1e-3 * rng.uniform(-1, 1, (3, 3)) if perturb else 0.0)


def test_kinematics_dynamics_oracle_vs_reference_build(sys_oracle, ref):
    rng = np.random.default_rng(7)
    for i in range(400):
        rho = (0.0, 2.0, 0.5)[i % 3]
        tw, R = rng.uniform(-1, 1, 6), _rand_rot(rng, i % 5 == 0)
        pd_o, rd_o = sys_oracle.kinematics_dynamics(rho, tw, R)
        pd_r, rd_r = ref.kin_dynamics(rho, tw, R)
        assert np.array_equal(pd_o, pd_r) and np.array_equal(rd_o, rd_r), f"state {i}"
    # rho == 0 with a singular rotation: the reference's 0 * ((R R^T)^-1 - I) R is NaN
    # (FloatingBaseSystemKinematics.cpp:62-66), and so is the oracle; the CUDA backend documents
    # that it skips the inverse there (tests/test_gpu_sys.py pins that side)
    tw = np.array([0.1, -0.2, 0.3, 0.4, 0.5, -0.6])
    singular = np.array([[1.0, 2.0, 3.0], [2.0, 4.0, 6.0], [0.5, -1.0, 0.25]])
    _, rd_r = ref.kin_dynamics(0.0, tw, singular)
    _, rd_o = sys_oracle.kinematics_dynamics(0.0, tw, singular)
    assert np.isnan(rd_r).all() and np.isnan(np.asarray(rd_o)).all()


@pytest.mark.parametrize("dt,t0,tf", [(0.01, 0.0, 0.1), (0.01, 0.0, 0.105), (0.003, 0.2, 0.25),
                                      (0.1, 0.0, 0.05), (0.01, 0.0, 0.01), (0.02, 1.0, 1.14)])
def test_integrate_schedule_oracle_vs_reference_build(sys_oracle, ref, dt, t0, tf):
    """FixedStepIntegrator::integrate incl. its last-step quirk (FixedStepIntegrator.tpp:48-64)."""
    rng = np.random.default_rng(int(dt * 1e4 + tf * 1e3))
    for rho in (0.0, 1.5):
        tw, R, p = rng.uniform(-1, 1, 6), _rand_rot(rng, False), rng.normal(size=3)
        jv, jp = rng.normal(size=5), rng.normal(size=5)
        steps, po, ro, jo = sys_oracle.integrate(rho, dt, t0, tf, tw, p, R, jv, jp)
        ok, pr, rr, jr = ref.kin_integrate(rho, dt, t0, tf, tw, p, R, jv, jp)
        assert ok and steps > 0
        assert np.array_equal(po, pr) and np.array_equal(ro, rr) and np.array_equal(jo, jr)


def test_integrate_refusals_match(sys_oracle, ref):
    rng = np.random.default_rng(3)
    tw, R, p = rng.uniform(-1, 1, 6), _rand_rot(rng, False), rng.normal(size=3)
    assert ref.kin_integrate(0.0, 0.01, 1.0, 0.5, tw, p, R)[0] is False      # tf < t0
    assert sys_oracle.integrate(0.0, 0.01, 1.0, 0.5, tw, p, R)[0] == -1
    assert ref.kin_integrate(0.0, -0.01, 0.0, 0.5, tw, p, R)[0] is False     # dT <= 0
    assert sys_oracle.integrate(0.0, -0.01, 0.0, 0.5, tw, p, R)[0] == -1


# --- J^T * wrench accumulation of FloatingBaseDynamicalSystem::dynamics ----------------------------

@pytest.mark.parametrize("cps,ncols,het,with_base", [(2, 29, False, True), (4, 38, True, True),
                                                     (1, 6, False, False), (3, 12, True, True),
                                                     (2, 7, False, False)])
def test_generalized_force_oracle_vs_reference_build(sys_oracle, ref, cps, ncols, het, with_base):
    """src/System/src/FloatingBaseSystemDynamics.cpp compiled unmodified and run over a
    KinDynComputations TEST DOUBLE (identity mass matrix, injected Jacobians / bias forces / frame
    states): [baseAcceleration; jointAcceleration] = -h + sum_c J_c^T wrench_c."""
    rng = np.random.default_rng(1000 * cps + ncols)
    ns = 400
    n = ns * cps
    st = syn.make_states(n, seed=70 + cps, heterogeneous=het)
    J = rng.normal(size=(n, 6, ncols))
    base = rng.normal(size=(ns, ncols)) if with_base else None
    planes = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])
    o, wo = sys_oracle.generalized_force(cps, ncols, planes, J, base,
                                         param_planes=st["params"].T if het else None,
                                         uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True, nthreads=2)
    r, wr = ref.generalized_force(cps, ncols, st["twists"], st["poses"], st["null_poses"], J, base,
                                  params=st["params"] if het else None,
                                  uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True, nthreads=4)
    assert np.array_equal(o, r) and np.array_equal(wo.T, wr)


# --- the whole of dynamics(): -bias + J^T wrench + torques, (M + reg).llt().solve -------------------

@pytest.mark.parametrize("cps,ncols,het,with_tau,with_reg,spread", [
    (2, 29, False, True, False, 0.0), (2, 29, True, True, True, 1.0), (1, 6, False, False, False, 0.5),
    (4, 38, True, True, True, 0.5), (3, 12, False, True, False, 1.5), (2, 7, True, True, True, 0.0)])
def test_floating_base_dynamics_oracle_vs_reference_build(sys_oracle, ref, cps, ncols, het, with_tau,
                                                          with_reg, spread):
    """FloatingBaseSystemDynamics.cpp compiled unmodified, run over the KinDynComputations test double
    loaded with random symmetric positive definite mass matrices, bias forces, joint torques and
    (through setMassMatrixRegularization) a regularisation term.  Bit for bit: the stand-in Eigen
    evaluates LLT in the order the C oracle restates."""
    rng = np.random.default_rng(77 * cps + ncols)
    ns = 300
    n = ns * cps
    st = syn.make_states(n, seed=90 + cps, heterogeneous=het)
    J = rng.normal(size=(n, 6, ncols))
    bias = rng.normal(size=(ns, ncols)) * 20.0
    tau = rng.normal(size=(ns, ncols - 6)) * 5.0 if with_tau and ncols > 6 else None
    reg = None
    if with_reg:
        reg = np.diag(10.0 ** rng.uniform(-4, -2, ncols))
        reg[ncols - 1, 0] = reg[0, ncols - 1] = 1e-3
    M = syn.make_mass_matrices(ns, ncols, seed=11 + ncols, spread=spread)
    planes = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])
    o, wo = sys_oracle.floating_base_acceleration(cps, planes, J, bias, M, tau, reg,
                                                  param_planes=st["params"].T if het else None,
                                                  uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True,
                                                  nthreads=2)
    r, wr = ref.floating_base_dynamics(cps, st["twists"], st["poses"], st["null_poses"], J, bias, M, tau, reg,
                                       params=st["params"] if het else None,
                                       uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True, nthreads=4)
    assert np.isfinite(r).all()
    assert np.array_equal(o, r) and np.array_equal(wo.T, wr)


@pytest.mark.parametrize("cps,ncols,rho,het", [(2, 29, 0.0, False), (2, 29, 0.7, True), (1, 6, 0.3, False),
                                               (3, 12, 2.0, False), (4, 38, 0.01, True)])
def test_floating_base_euler_step_oracle_vs_reference_build(sys_oracle, ref, cps, ncols, rho, het):
    """ForwardEuler<FloatingBaseDynamicalSystem>(dT).integrate(0, dT) from the reference's own sources
    (ForwardEuler.tpp + FloatingBaseSystemDynamics.cpp over the test double): the acceleration at the old
    state, then x += dx * dT over the whole state tuple.  Bit for bit."""
    rng = np.random.default_rng(5 * cps + ncols)
    ns, dT = 200, 0.01
    st = syn.make_states(ns * cps, seed=33 + cps, heterogeneous=het)
    J = rng.normal(size=(ns * cps, 6, ncols))
    bias = rng.normal(size=(ns, ncols)) * 20.0
    tau = rng.normal(size=(ns, ncols - 6)) if ncols > 6 else None
    M = syn.make_mass_matrices(ns, ncols, seed=3 + ncols, spread=0.5)
    nu = rng.normal(size=(ns, ncols))
    jp = rng.normal(size=(ns, ncols - 6)) if ncols > 6 else None
    p = rng.normal(size=(ns, 3))
    R = np.stack([_rand_rot(rng, i % 3 == 0) for i in range(ns)])
    planes = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])
    acc = sys_oracle.floating_base_acceleration(cps, planes, J, bias, M, tau,
                                                param_planes=st["params"].T if het else None,
                                                uniform=syn.REFERENCE_TEST_PARAMS, nthreads=2)
    v, q, pp, RR = sys_oracle.floating_base_euler_step(rho, dT, acc, nu, jp, p, R, nthreads=2)
    racc, rv, rq, rp, rR = ref.floating_base_euler_step(cps, st["twists"], st["poses"], st["null_poses"], J, bias, M,
                                                        rho, dT, nu, jp, p, R, joint_torques=tau,
                                                        params=st["params"] if het else None,
                                                        uniform=syn.REFERENCE_TEST_PARAMS, nthreads=4)
    assert np.array_equal(acc, racc) and np.array_equal(v, rv) and np.array_equal(pp, rp) and np.array_equal(RR, rR)
    if jp is not None:
        assert np.array_equal(q, rq)
    # the step really moved the state, and positions used the OLD velocities
    assert np.array_equal(pp, p + nu[:, :3] * dT)


# --- integrate -> contact model rollout ------------------------------------------------------------

@pytest.mark.parametrize("rho", [0.0, 2.0])
def test_rollout_oracle_vs_reference_build(sys_oracle, ref, rho):
    nr, feet, H, dT = 37, 2, 25, 0.01
    chains = nr * feet
    st = syn.make_states(chains, seed=50, heterogeneous=True)
    tw = np.random.default_rng(3).uniform(-1, 1, (H, chains, 6))
    r = ref.rollout(tw, st["poses"], st["null_poses"], dT, rho, params=st["params"], mask=7, nthreads=4)
    o = sys_oracle.rollout(nr, feet, H, dT, rho, np.ascontiguousarray(tw.reshape(H * chains, 6).T),
                           np.ascontiguousarray(st["poses"][:, :3].T),
                           np.ascontiguousarray(st["poses"][:, 3:].T),
                           np.ascontiguousarray(st["null_poses"].T),
                           param_planes=np.ascontiguousarray(st["params"].T), mask=7,
                           wrench_ref=np.zeros(6), weights=np.ones(2), nthreads=2)
    assert np.array_equal(o["wrench"].T, r["wrench"])
    assert np.array_equal(o["autodyn"].T, r["autodyn"])
    assert np.array_equal(o["ctrl"], r["ctrl"])
    assert np.array_equal(o["pos"].T, r["final_poses"][:, :3])
    assert np.array_equal(o["rot"].T, r["final_poses"][:, 3:])


# --- how much can the part the stand-in leaves open matter? ---------------------------------------

def test_evaluation_order_and_fma_choices_move_results_far_below_tolerance(ref):
    """The stand-in Eigen is not Eigen: it fixes one association of the 3-term inner sums and the
    default build forbids FMA contraction.  libblf_reference_alt.so is the same reference source built
    with the OTHER choices (tree-shaped sums as Eigen's unrolled reductions, -ffp-contract=fast -mfma).
    The two builds differ -- most outputs in the last bits -- but norm-wise by < 1e-13 (measured:
    8e-15), three orders of magnitude under the 1e-12 parity tolerance."""
    from parity import block_rel_err
    if not os.path.exists(ref.ALT_LIB_PATH) and not ref.reference_sources_present():
        pytest.skip("alternative reference build not available")
    st = syn.make_states(200_000, seed=49, heterogeneous=True)
    a = ref.eval_batch_states(st, MASK_ALL, nthreads=4)
    b = ref.eval_batch_states_alt(st, MASK_ALL, nthreads=4)
    differing = 0
    for key in ("wrench", "autodyn", "ctrl", "regressor"):
        differing += int((a[key] != b[key]).any(axis=1).sum())
        assert block_rel_err(b[key], a[key], key).max() < 1e-13, key
    assert differing > 1000          # the alternative build really does round differently
    assert np.array_equal(a["ctrl"], b["ctrl"]) or block_rel_err(b["ctrl"], a["ctrl"], "ctrl").max() < 1e-13


# --- special values: the restatement must propagate them exactly as the reference's code does ------

def test_special_values_oracle_vs_reference_build(oracle, ref):
    """Infinities, NaNs, signed zeros, denormals and huge/tiny magnitudes sprinkled over otherwise
    ordinary states: same bits out of the C restatement and the reference build (NaN == NaN)."""
    n = 20_000
    st = syn.make_states(n, seed=99, heterogeneous=True)
    rng = np.random.default_rng(99)
    specials = np.array([np.inf, -np.inf, np.nan, 0.0, -0.0, 5e-324, -2.2e-308, 1e300, -1e300, 1e-300,
                         1.7976931348623157e308])
    for key, width in (("twists", 6), ("poses", 12), ("null_poses", 12), ("params", 4)):
        a = st[key]
        hit = rng.random((n, width)) < 0.03
        a[hit] = rng.choice(specials, size=int(hit.sum()))
    with np.errstate(all="ignore"):
        a = oracle.eval_batch_states(st, MASK_ALL, nthreads=4)
        b = ref.eval_batch_states(st, MASK_ALL, nthreads=4)
    for key in ("wrench", "autodyn", "ctrl", "regressor"):
        assert np.array_equal(a[key], b[key], equal_nan=True), key
        finite = np.isfinite(a[key])
        assert np.array_equal(np.signbit(a[key][finite]), np.signbit(b[key][finite])), key
    # the structural zeros of the control matrix stay +0.0 whatever the inputs (never written)
    from parity import CTRL_STRUCTURAL_ZERO
    z = b["ctrl"][:, CTRL_STRUCTURAL_ZERO]
    assert np.all(z == 0.0) and not np.signbit(z).any()
