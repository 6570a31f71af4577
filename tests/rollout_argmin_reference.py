"""The selection rule and the cost tolerance of the rollout-cost arg-min, in plain Python, for the
tests of blf_ccm_rollout_cost_argmin_soa and blf_ccm_argmin_pairs.

Selection (what the device's (cost, index) pair must be):
  - NaN never wins; +inf is comparable and can win;
  - among equal costs (-0.0 == +0.0) the lowest index wins;
  - (+inf, -1) when nothing is comparable or the batch is empty;
  - the returned cost has the bits of the winning entry.
blf_ccm_argmin_pairs also skips every pair whose index is negative.
"""
from __future__ import annotations

import numpy as np

from parity import TOL


def best_of_pairs(cost, idx):
    """(cost, index) the rule selects among the pairs (cost[j], idx[j]); pairs with idx < 0 skipped."""
    c = np.asarray(cost, dtype=np.float64).reshape(-1)
    i = np.asarray(idx, dtype=np.int64).reshape(-1)
    ok = (i >= 0) & ~np.isnan(c)
    if not ok.any():
        return float("inf"), -1
    m = c[ok].min()
    cand = np.nonzero(ok & (c == m))[0]
    j = cand[np.argmin(i[cand])]
    return float(c[j]), int(i[j])


def expected_best(cost, index_base=0):
    """The pair for a batch whose rollout r has cost[r] and global index index_base + r."""
    c = np.asarray(cost, dtype=np.float64).reshape(-1)
    return best_of_pairs(c, np.int64(index_base) + np.arange(c.size, dtype=np.int64))


def bits(x) -> int:
    return int(np.float64(x).view(np.uint64))


def cost_scale(wrench, rollout_len, wrench_ref, weights):
    """Per rollout, sum_e wf (|F_e| + |F_ref|)^2 + wt (|T_e| + |T_ref|)^2: the magnitude the rounding
    error of any evaluation of the cost is proportional to (not the cost itself, which cancels
    when F ~ F_ref)."""
    w = np.asarray(wrench, dtype=np.float64).reshape(-1, 6)
    ref = np.asarray(wrench_ref, dtype=np.float64)
    f = np.linalg.norm(w[:, :3], axis=1) + np.linalg.norm(ref[:3])
    t = np.linalg.norm(w[:, 3:], axis=1) + np.linalg.norm(ref[3:])
    per = weights[0] * f * f + weights[1] * t * t
    return per.reshape(-1, rollout_len).sum(axis=1)


def assert_costs_within(got, ref, scale, what=""):
    got, ref = np.asarray(got), np.asarray(ref)
    assert np.all(np.isfinite(got)), f"{what}: non-finite cost"
    err = np.abs(got - ref)
    bad = np.nonzero(err > TOL * scale)[0]
    assert bad.size == 0, (f"{what}: rollout {bad[0]} of {got.size}: cost {got[bad[0]]!r}, reference "
                           f"{ref[bad[0]]!r}, error {err[bad[0]]:.3e} > TOL x {scale[bad[0]]:.3e}")
