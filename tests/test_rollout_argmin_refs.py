"""CPU checks of the references the rollout-cost arg-min tests rely on: exact_rollout_cost (exact
Fractions over the golden states) against the C oracle's ccmo_rollout_cost, and the selection
rule of expected_best / best_of_pairs on hand-made vectors."""
import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from oracle.exact_golden import exact_eval, exact_rollout_cost
from rollout_argmin_reference import assert_costs_within, best_of_pairs, bits, cost_scale, expected_best

REF_W = np.array([1.0, -2.0, 30.0, 0.1, 0.2, -0.3])
WTS = np.array([1.0, 25.0])
INF, NAN = float("inf"), float("nan")


def _batch(golden, rollout_len, n_rollouts, seed):
    """Every golden state at least once, in a seeded order, repeated to n_rollouts x rollout_len."""
    n = rollout_len * n_rollouts
    rows = np.random.default_rng(seed).permutation(np.resize(np.arange(golden["twists"].shape[0]), n))
    return {k: golden[k][rows] for k in ("twists", "poses", "null_poses", "params")}


@pytest.mark.parametrize("rollout_len,n_rollouts", [(1, 201), (33, 7), (256, 2)])
@pytest.mark.parametrize("het", [False, True], ids=["uniform", "per-contact"])
def test_exact_rollout_cost_vs_c_oracle(golden, oracle, rollout_len, n_rollouts, het):
    st = _batch(golden, rollout_len, n_rollouts, seed=rollout_len)
    params = st["params"] if het else np.array(syn.REFERENCE_TEST_PARAMS)
    exact = exact_rollout_cost(st, rollout_len, REF_W, WTS, params)
    w = oracle.eval_batch_aos(st["twists"], st["poses"], st["null_poses"], params=st["params"] if het else None,
                              uniform=None if het else params, mask=1)["wrench"]
    ref = oracle.rollout_cost(w, rollout_len, REF_W, WTS)
    assert exact.shape == (n_rollouts,)
    assert_costs_within(ref, exact, cost_scale(w, rollout_len, REF_W, WTS), "C oracle vs exact")


def test_exact_rollout_cost_rounds_once(golden):
    """A rollout of one state with F_ref = 0 and weights (1, 0) costs |F|^2 rounded once; the all-zero
    state and zero parameters cost exactly 0."""
    st = {k: golden[k][[0, 1, 5]] for k in ("twists", "poses", "null_poses", "params")}
    got = exact_rollout_cost(st, 1, np.zeros(6), [1.0, 0.0], st["params"])
    f = exact_eval(st["twists"][0], st["poses"][0], st["null_poses"][0], st["params"][0])["wrench"][:3]
    assert got[0] == float(sum(x * x for x in f)) and got[0] > 0
    assert got[1] == 0.0 and got[2] == 0.0
    # a uniform parameter tuple is the same as that tuple on every state
    prm = np.array(syn.REFERENCE_TEST_PARAMS)
    a = exact_rollout_cost(st, 3, REF_W, WTS, prm)
    b = exact_rollout_cost(st, 3, REF_W, WTS, np.tile(prm, (3, 1)))
    assert a.shape == (1,) and a[0] == b[0]


def test_expected_best_selection_rule():
    eb = expected_best
    assert eb([3.0, 1.0, 2.0]) == (1.0, 1)
    assert eb([3.0, 1.0, 1.0, 0.5, 0.5], 10) == (0.5, 13)            # lowest index among ties
    assert eb([NAN, 2.0, NAN, 2.0]) == (2.0, 1)                       # NaN never wins
    assert eb([NAN, INF, NAN, INF], 7) == (INF, 8)                    # +inf is comparable
    assert eb([INF, 5.0]) == (5.0, 1)
    assert eb([NAN, NAN]) == (INF, -1) and eb([]) == (INF, -1)
    c, i = eb([1.0, -0.0, 0.0])                                       # -0.0 == +0.0: index 1 and its bits
    assert i == 1 and bits(c) == bits(-0.0)
    c, i = eb([1.0, 0.0, -0.0])
    assert i == 1 and bits(c) == bits(0.0)
    base = 2 ** 40 + 3
    assert eb([2.0, 1.0, 1.0], base) == (1.0, base + 1)
    assert eb(np.full(5000, 4.0), 2 ** 40) == (4.0, 2 ** 40)


def test_best_of_pairs_selection_rule():
    bp = best_of_pairs
    assert bp([3.0, 1.5, 1.5, 2.0], [5, 9, 4, 1]) == (1.5, 4)         # lowest index, not first position
    assert bp([-5.0, 1.0, -9.0], [-1, 3, -2]) == (1.0, 3)             # negative indices skipped
    assert bp([-5.0, NAN], [-1, 2]) == (INF, -1)
    assert bp([], []) == (INF, -1)
    c, i = bp([0.0, -0.0], [8, 2])
    assert i == 2 and bits(c) == bits(-0.0)
    c, i = bp([-0.0, 0.0], [8, 2])
    assert i == 2 and bits(c) == bits(0.0)
    assert bp([NAN, INF], [0, 1]) == (INF, 1)
