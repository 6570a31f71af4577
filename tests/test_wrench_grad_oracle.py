"""CPU checks of the references for the wrench's reverse mode (tests/wrench_grad_reference.py): the
exact forward-mode Jacobians pin the golden fixture, the float64 torch restatement agrees with them
and its forward with the C oracle, and the (spring, damper) columns are the regressor's."""
import os

import numpy as np

import wrench_grad_reference as ref
from parity import assert_parity

TOL = 1e-12


def test_exact_jacobians_reproduce_the_golden_fixture():
    gd = ref.load_golden()
    g = dict(np.load(os.path.join(ref.ROOT, "tests", "golden", "ccm_exact_golden.npz")))
    assert gd["jacobian"].shape == (201, 6, ref.NCOLS)
    for key in ("twists", "poses", "null_poses", "params"):
        assert np.array_equal(gd[key], g[key])
    assert list(gd["live_planes"]) == ref.LIVE_PLANES
    for i in range(gd["jacobian"].shape[0]):
        J = ref.exact_jacobian(gd["twists"][i], gd["poses"][i], gd["null_poses"][i], gd["params"][i])
        assert np.array_equal(np.array([[float(v) for v in row] for row in J]), gd["jacobian"][i]), i


def test_exact_jacobian_edge_states():
    gd = ref.load_golden()
    J = gd["jacobian"]
    c_r22 = ref.LIVE_PLANES.index(17)
    assert gd["poses"][3, 11] == 0.0 and gd["poses"][4, 11] == 0.0       # R22 = +0, -0
    assert np.all(J[3:5, :, c_r22] == 0.0)                                # sgn(+-0) = 0
    assert np.all(J[3:5] == 0.0)                                          # |R22| = 0 scales everything
    assert gd["poses"][2, 11] == -1.0 and np.any(J[2, :, c_r22] != 0.0)   # inverted foot
    assert np.any(J[8] != 0.0)                                            # pose == null pose


def test_torch_restatement_forward_matches_the_c_oracle(oracle):
    import torch
    from bipedal_locomotion_framework_b200 import synthetic as syn
    for het in (False, True):
        st = syn.make_states(4096, seed=77 + het, heterogeneous=het)
        prm = st["params"] if het else np.tile(syn.REFERENCE_TEST_PARAMS, (st["n"], 1))
        planes = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])
        got = ref.torch_wrench(torch.from_numpy(planes), torch.from_numpy(prm.T.copy())).numpy().T
        want = oracle.eval_batch_aos(st["twists"], st["poses"], st["null_poses"], prm, None, 1)["wrench"]
        assert_parity(got, want, "wrench", what=f"het={het} ")


def test_torch_restatement_gradient_matches_the_exact_goldens():
    gd = ref.load_golden()
    planes, prm = ref.golden_planes(gd)
    n = planes.shape[1]
    rng = np.random.default_rng(3)
    for trial in range(7):
        # six one-hot cotangents give the Jacobian rows, the seventh is random
        g = np.zeros((6, n))
        if trial < 6:
            g[trial] = 1.0
        else:
            g = rng.uniform(-1, 1, (6, n))
        got_x, got_p = ref.torch_vjp(planes, prm, g)
        want_x, want_p = ref.golden_vjp(gd, g)
        assert np.all(got_x[list(ref.DEAD_PLANES)] == 0.0)
        mag_x, mag_p = ref.operand_magnitude(planes, prm, g)
        err = ref.vjp_errors(got_x, got_p, want_x, want_p, mag_x, mag_p)
        assert err.max() <= TOL, (trial, int(err.argmax()), err.max())


def test_spring_and_damper_columns_are_the_regressor(oracle):
    gd = ref.load_golden()
    reg = oracle.eval_batch_aos(gd["twists"], gd["poses"], gd["null_poses"], gd["params"], None,
                                oracle.REGRESSOR, 1)["regressor"].reshape(-1, 6, 2)
    J = gd["jacobian"]
    ck, cb = ref.NCOLS - 2, ref.NCOLS - 1
    floor = np.full(J.shape[0], 1e-300)
    floor[8] = 1e-6  # pose == null pose: the torque block cancels to exactly 0 (see test_gpu_parity.py)
    got = np.concatenate([J[:, :, ck:ck + 1], J[:, :, cb:cb + 1]], axis=2).reshape(-1, 12)
    assert_parity(got, reg.reshape(-1, 12), "regressor", floor=floor)
    # and for a random cotangent, gbar . column
    rng = np.random.default_rng(5)
    g = rng.uniform(-1, 1, (6, J.shape[0]))
    _, gp = ref.golden_vjp(gd, g)
    want = np.einsum("nrc,rn->cn", reg, g)
    assert np.allclose(gp[2:4], want, rtol=1e-12, atol=1e-12 * np.abs(reg).max())
