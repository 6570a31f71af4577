"""CPU checks of the references for the rollout cost's reverse mode (tests/rollout_grad_reference.py):
the golden fixture is what the 80-digit references compute, the float64 torch restatement (a) agrees
with forward mode on duals (b) at short horizons and with 80-digit central differences (c) at
H = 100, its forward cost is the C oracle's, and (c)'s chain cost is mp_rollout's.

WORST_F64 records the worst norm-wise relative error (per chain and gradient group) float64 reaches
at each horizon of the fixture, measured with these references; the GPU tests' tolerances rest on it."""
import numpy as np
import pytest

import rollout_grad_reference as ref

# horizon -> the worst relative error of (a) measured against (b) / (c), and the bound asserted
WORST_F64 = {1: 5.3e-16, 3: 1.6e-15, 5: 4.1e-16, 6: 4.0e-16, 100: 1.0e-15}
BOUND_SHORT = 1e-14
BOUND_LONG = 1e-12


@pytest.fixture(scope="module")
def golden():
    return ref.load_golden()


@pytest.mark.parametrize("row", ref.SHORT_CASES, ids=[r[0] for r in ref.SHORT_CASES])
def test_torch_restatement_against_forward_mode(golden, row):
    case, dT, rho = ref.case_from_row(row)
    g, _ = ref.torch_grads(case, dT, rho)
    dual = golden[row[0] + "/dual"]
    worst = 0.0
    for c in range(case["n_rollouts"] * case["feet"]):
        got = ref.chain_vector(g, case, c) / case["grad_cost"][c // case["feet"]]
        err = ref.group_errors(got, dual[c], case["horizon"])
        worst = max(worst, *err.values())
    assert worst <= BOUND_SHORT, (row[0], worst)
    assert worst <= 4 * WORST_F64[case["horizon"]], (row[0], worst, "the record of WORST_F64 is stale")


def test_forward_mode_reproduces_the_golden_fixture(golden):
    row = ref.SHORT_CASES[2]
    case, dT, rho = ref.case_from_row(row)
    for c in range(case["n_rollouts"] * case["feet"]):
        d = ref.dual_chain_gradient(ref.chain_inputs(case, c), case["horizon"], dT, rho)
        assert np.array_equal(d, golden[row[0] + "/dual"][c]), c


def test_edge_chains_are_in_the_cases():
    for row in ref.SHORT_CASES:
        case, _, _ = ref.case_from_row(row)
        assert case["rot"][8, 1] < 0.0                                  # the inverted foot
    case, _, _ = ref.case_from_row(ref.SHORT_CASES[0])
    assert np.array_equal(case["null"][:, 0], np.concatenate([case["pos"][:, 0], case["rot"][:, 0]]))


@pytest.mark.parametrize("row", ref.LONG_CASES, ids=[r[0] for r in ref.LONG_CASES])
def test_torch_restatement_against_central_differences(golden, row):
    case, dT, rho = ref.case_from_row(row)
    g, _ = ref.torch_grads(case, dT, rho)
    coords, fd = golden[row[0] + "/coords"], golden[row[0] + "/fd"]
    worst = 0.0
    for c in range(case["n_rollouts"] * case["feet"]):
        got = ref.chain_vector(g, case, c)[coords[c]] / case["grad_cost"][c // case["feet"]]
        scale = np.linalg.norm(ref.chain_vector(g, case, c)) / case["grad_cost"][c // case["feet"]]
        # sampled coordinates: each against the chain's whole gradient norm (coordinates can vanish)
        worst = max(worst, np.max(np.abs(got - fd[c])) / scale)
    assert worst <= BOUND_LONG, (row[0], worst)
    assert worst <= 4 * WORST_F64[100], (row[0], worst, "the record of WORST_F64 is stale")


@pytest.mark.parametrize("rho", [0.0, 0.5])
def test_torch_forward_cost_matches_the_c_oracle(rho):
    import torch
    from oracle import sys_oracle
    case = ref.make_case(8, 2, 12, seed=31, het=True, inverted=True, at_null=True)
    args = (case["n_rollouts"], case["feet"], case["horizon"], 0.01, rho)
    want = sys_oracle.rollout(*args, case["twist"], case["pos"], case["rot"], case["null"],
                              param_planes=case["params"], wrench_ref=ref.REF, weights=ref.WEIGHTS)["cost"]
    t = lambda k: torch.tensor(case[k], dtype=torch.float64)
    got = ref.torch_rollout_cost(*args, t("twist"), t("pos"), t("rot"), t("null"), t("params"),
                                 ref.REF, ref.WEIGHTS).numpy()
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)


def test_central_difference_cost_is_mp_rollout():
    from oracle.exact_golden_sys import mp_rollout
    case = ref.make_case(1, 2, 3, seed=41, het=True, inverted=True)
    out = mp_rollout(1, 2, 3, 0.01, 0.5, case["twist"], case["pos"], case["rot"], case["null"], case["params"],
                     ref.REF, ref.WEIGHTS)
    for c in range(2):
        got = float(ref.mp_chain_cost(ref.chain_inputs(case, c), 3, 0.01, 0.5))
        assert got == out["chain_cost"][c]
