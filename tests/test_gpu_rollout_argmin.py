"""GPU tests of the sampling-MPC rollout cost and its arg-min: blf_ccm_rollout_cost_argmin_soa
(ccm_soa_kernel<OUT, HET, COST=true> + ccm_cost_reduce_kernel), blf_ccm_argmin_pairs, and the
reduction launch of blf_ccm_rollout_integrate_cost's two-launch forms.

  A. every cost instance (out_mask 0..7 x uniform / per-contact parameters) on golden states,
     against exact costs and exact outputs
  B. every tile alignment of a rollout (lengths 1 .. 4097, batches of 0, 1 and 31 rollouts mod 32)
  C. planted minima and exact ties at every level of the reduction: lanes, warps, blocks, the
     last-block combine and the second grid-stride pass (past 8192 x 128 rollouts)
  D. NaN and +inf costs
  E. windows combined with blf_ccm_argmin_pairs, as a multi-window or multi-rank caller does
  F. blf_ccm_argmin_pairs on its own
  G. scratch growth, guard bands, determinism
  H. the same reduction fed by the fused rollout (fixed_count) past one grid-stride pass

What may be bit for bit: a tile's partial is the xor butterfly over its 32 lanes (lanes outside the
rollout add +0.0) and the reduction adds a rollout's partials in tile order from +0.0, so a
rollout's cost has the same bits between calls only where its contacts sit at the same offsets
mod 32.  Costs are otherwise held to TOL x sum_e wf (|F_e| + |F_ref|)^2 + wt (|T_e| + |T_ref|)^2,
and the arg-min is held bit for bit to the selection rule applied to the device's own costs.
A planted rollout (R(2,2) = 0, or spring = damper = 0, with F_ref = 0) costs exactly +0.0."""
import ctypes as C

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from oracle.exact_golden import exact_eval_rounded, exact_rollout_cost
from parity import assert_ctrl_structure, assert_parity
from rollout_argmin_reference import assert_costs_within, best_of_pairs, bits, cost_scale, expected_best

pytestmark = pytest.mark.gpu

SENTINEL = -7.25e300
REF_W = np.array([1.0, -2.0, 30.0, 0.1, 0.2, -0.3])
ZERO_W = np.zeros(6)
WTS = np.array([1.0, 25.0])
REF_PARAMS = np.array(syn.REFERENCE_TEST_PARAMS)
INF, NAN = float("inf"), float("nan")
R22 = 17                      # plane of the pose's R(2,2)
PASS = 8192 * 128             # rollouts per grid-stride pass of ccm_cost_reduce_kernel
BIG_BASE = 2 ** 40 + 3


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


@pytest.fixture(scope="module")
def lib(torch):
    from bipedal_locomotion_framework_b200 import _capi
    return _capi.lib()


def _new_handle():
    from bipedal_locomotion_framework_b200.contact_models import _Handle
    h = _Handle(0)
    h.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    return h


@pytest.fixture(scope="module")
def handle(torch):
    h = _new_handle()
    yield h
    h.close()


def _pp(t, count):
    """Plane-pointer array of a (count, n) tensor or a list of 1-D tensors / None."""
    if t is None:
        return None
    return (C.c_void_p * count)(*[None if t[i] is None else t[i].data_ptr() for i in range(count)])


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _stream(torch):
    return torch.cuda.current_stream().cuda_stream


def _rollout(torch, lib, h, planes, rollout_len, prm=None, mask=0, out=None, ref=REF_W, wts=WTS,
             index_base=0, cost_ptr=-1, best_ptr=None, n_rollouts=None):
    """One blf_ccm_rollout_cost_argmin_soa call.  cost_ptr: -1 = a fresh SENTINEL-filled tensor,
    None = NULL, else a device address.  Returns (cost tensor or None, best tensor or None)."""
    n = planes.shape[1] if hasattr(planes, "shape") else next(p for p in planes if p is not None).shape[0]
    nr = n // rollout_len if n_rollouts is None else n_rollouts
    cost = None
    if cost_ptr == -1:
        cost = torch.full((nr,), SENTINEL, dtype=torch.float64, device="cuda")
        cost_ptr = cost.data_ptr()
    best = None
    if best_ptr is None:
        best = torch.empty(2, dtype=torch.int64, device="cuda")
        best_ptr = best.data_ptr()
    out = out or {}
    refa, wa = np.ascontiguousarray(ref, dtype=np.float64), np.ascontiguousarray(wts, dtype=np.float64)
    rc = lib.blf_ccm_rollout_cost_argmin_soa(h.ptr, nr, rollout_len, _pp(planes, 30), _pp(prm, 4), mask,
                                             _pp(out.get("wrench"), 6), _pp(out.get("autodyn"), 6),
                                             out["ctrl"].data_ptr() if out.get("ctrl") is not None else None,
                                             refa.ctypes.data, wa.ctypes.data, int(index_base), cost_ptr,
                                             best_ptr, _stream(torch))
    assert rc == 0, lib.blf_ccm_last_error().decode()
    return cost, best


def _decode(best):
    """(cost, index, cost bits) of a 16-byte pair."""
    b = best.cpu().numpy().astype(np.int64)
    return float(b[:1].view(np.float64)[0]), int(b[1]), int(b[:1].view(np.uint64)[0])


def _assert_best(best, want, what):
    c, i, cb = _decode(best)
    wc, wi = want
    assert (i, cb) == (wi, bits(wc)), f"{what}: best ({c!r}, {i}), expected ({wc!r}, {wi})"


def _states_planes(torch, st):
    planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
    prm = _dev(torch, st["params"].T) if st.get("params") is not None else None
    return planes, prm


def _outputs(torch, n):
    return {"wrench": torch.full((6, n), SENTINEL, dtype=torch.float64, device="cuda"),
            "autodyn": torch.full((6, n), SENTINEL, dtype=torch.float64, device="cuda"),
            "ctrl": torch.full((n * 36,), SENTINEL, dtype=torch.float64, device="cuda")}


# --- A. every instance against exact costs -----------------------------------------------------------

GOLDEN_SHAPES = ((256, 12), (33, 97))   # (rollout_len, n_rollouts)


@pytest.fixture(scope="module")
def golden_batches(golden):
    """Batches assembled from the golden states (each at least once, seeded order, repeated), with
    their exact costs and exact outputs, for uniform and per-contact parameters."""
    ng = golden["twists"].shape[0]
    uni = [exact_eval_rounded(golden["twists"][i], golden["poses"][i], golden["null_poses"][i], REF_PARAMS)
           for i in range(ng)]
    exact_uni = {k: np.stack([r[k] for r in uni]) for k in ("wrench", "autodyn", "ctrl")}
    out = {}
    for L, nr in GOLDEN_SHAPES:
        rows = np.random.default_rng(L).permutation(np.resize(np.arange(ng), L * nr))
        st = {k: golden[k][rows] for k in ("twists", "poses", "null_poses", "params")}
        for het in (False, True):
            params = st["params"] if het else REF_PARAMS
            ref = {k: (golden[k] if het else exact_uni[k])[rows] for k in ("wrench", "autodyn", "ctrl")}
            out[L, het] = {"states": {**st, "params": st["params"] if het else None}, "ref": ref,
                           "cost": exact_rollout_cost(st, L, REF_W, WTS, params),
                           "scale": cost_scale(ref["wrench"], L, REF_W, WTS)}
    return out


@pytest.mark.parametrize("het", [False, True], ids=["uniform", "per-contact"])
@pytest.mark.parametrize("mask", range(8))
def test_every_instance_vs_exact(torch, lib, handle, golden_batches, mask, het):
    """CostLaunch<mask, het> at rollout_len 256 and 33: costs against exact Fractions, requested
    outputs against the exact outputs, unrequested planes untouched, and cost = NULL giving the
    same best bits."""
    for L, nr in GOLDEN_SHAPES:
        gb = golden_batches[L, het]
        what = f"mask {mask} {'per-contact' if het else 'uniform'} L={L}"
        planes, prm = _states_planes(torch, gb["states"])
        n = L * nr
        out = _outputs(torch, n)
        cost, best = _rollout(torch, lib, handle, planes, L, prm, mask, out, index_base=1000)
        c = cost.cpu().numpy()
        assert_costs_within(c, gb["cost"], gb["scale"], what)
        _assert_best(best, expected_best(c, 1000), what)
        got = {"wrench": out["wrench"].cpu().numpy().T, "autodyn": out["autodyn"].cpu().numpy().T,
               "ctrl": out["ctrl"].cpu().numpy().reshape(n, 36)}
        for bit, key in ((1, "wrench"), (2, "autodyn"), (4, "ctrl")):
            if mask & bit:
                assert_parity(got[key], gb["ref"][key], key, what=what + " ")
            else:
                assert np.all(got[key] == SENTINEL), f"{what}: {key} written though not requested"
        if mask & 4:
            assert_ctrl_structure(got["ctrl"])
        _, best_nc = _rollout(torch, lib, handle, planes, L, prm, mask, out, index_base=1000, cost_ptr=None)
        assert torch.equal(best_nc, best), f"{what}: cost = NULL changes best"


# --- B. tile alignments -------------------------------------------------------------------------------

ALIGN_LENS = (1, 2, 3, 5, 31, 32, 33, 63, 64, 65, 255, 256, 257, 1000, 4097)


def _align_counts(L):
    base = 4096 if L <= 5 else (256 if L <= 65 else 32)
    return (base, base + 1, base + 31)        # n_rollouts mod 32 = 0, 1, 31


@pytest.mark.parametrize("het", [False, True], ids=["uniform", "per-contact"])
@pytest.mark.parametrize("rollout_len", ALIGN_LENS)
def test_alignment_sweep_vs_oracle(torch, lib, handle, oracle, rollout_len, het):
    """Every rollout of the batch against the C oracle's wrench + rollout_cost; best bit for bit the
    selection rule on the device's own costs; masks 0 and 7 give the same cost bits."""
    L = rollout_len
    for nr in _align_counts(L):
        st = syn.make_states(nr * L, seed=1000 + L * 7 + nr, heterogeneous=het)
        planes, prm = _states_planes(torch, st)
        w = oracle.eval_batch_states(st, mask=1, nthreads=8)["wrench"]
        ref = oracle.rollout_cost(w, L, REF_W, WTS)
        scale = cost_scale(w, L, REF_W, WTS)
        first = None
        for mask in (0, 7):
            what = f"L={L} n_rollouts={nr} mask={mask} {'per-contact' if het else 'uniform'}"
            out = _outputs(torch, nr * L) if mask else None
            cost, best = _rollout(torch, lib, handle, planes, L, prm, mask, out)
            c = cost.cpu().numpy()
            assert_costs_within(c, ref, scale, what)
            _assert_best(best, expected_best(c), what)
            if first is None:
                first = c
            else:
                assert np.array_equal(c.view(np.uint64), first.view(np.uint64)), f"{what}: cost bits depend on the mask"


# --- C. planted minima across every reduction level ---------------------------------------------------

def _plant_sites(nr):
    return [0, 31, 32, 127, 128, 8191 * 128, PASS - 1, PASS, PASS + 1, nr - 1]


def _planter(torch, planes, prm, L, het):
    """plant(r, on): rollout r costs exactly +0.0 with F_ref = 0 (R(2,2) = 0 on its contacts, or
    spring = damper = 0 with per-contact parameters); on=False restores it."""
    keep = {}

    def plant(r, on):
        sl = slice(r * L, (r + 1) * L)
        tgt = [prm[2], prm[3]] if het else [planes[R22]]
        if on:
            keep[r] = [t[sl].clone() for t in tgt]
            for t in tgt:
                t[sl] = 0.0
        else:
            for t, v in zip(tgt, keep.pop(r)):
                t[sl] = v
    return plant


def _check_planted(torch, cost, planted, what):
    pl = torch.tensor(sorted(planted), dtype=torch.int64, device="cuda")
    z = cost[pl]
    assert bool((z == 0).all()) and not bool(torch.signbit(z).any()), f"{what}: a planted cost is not +0.0"
    mask = torch.ones_like(cost, dtype=torch.bool)
    mask[pl] = False
    assert bool((cost[mask] > 0).all()), f"{what}: an unplanted cost is not > 0 (invalid data)"


@pytest.mark.parametrize("het", [False, True], ids=["R22=0", "spring=damper=0"])
@pytest.mark.parametrize("rollout_len", [1, 3])
def test_planted_minima_every_reduction_level(torch, lib, handle, rollout_len, het):
    """2^20 + 4099 rollouts (two grid-stride passes of the reduction): exact +0.0 minima planted at
    lane, warp, block, last-block and second-pass boundaries.  For each k the sites k.. are
    planted, so site k must win against exact ties at every higher site, whatever level they meet
    at; index_base up to past 32 bits."""
    L, nr = rollout_len, PASS + 4099
    planes, prm = syn.make_planes_torch(nr * L, torch.device("cuda", 0), seed=70 + L, heterogeneous=het)
    plant = _planter(torch, planes, prm, L, het)
    sites = _plant_sites(nr)
    for r in sites:
        plant(r, True)
    for k, lowest in enumerate(sites):
        planted = sites[k:]
        for base in (0, 1000, BIG_BASE):
            what = f"L={L} planted {planted} index_base={base}"
            cost, best = _rollout(torch, lib, handle, planes, L, prm if het else None, ref=ZERO_W,
                                  index_base=base)
            if base == 0:
                _check_planted(torch, cost, planted, what)
            _assert_best(best, (0.0, lowest + base), what)
        plant(lowest, False)
    cost, best = _rollout(torch, lib, handle, planes, L, prm if het else None, ref=ZERO_W)
    c = cost.cpu().numpy()
    assert np.all(c > 0)
    _assert_best(best, expected_best(c), f"L={L} nothing planted")


# --- D. non-finite costs ------------------------------------------------------------------------------

def test_non_finite_costs(torch, lib, handle):
    """NaN costs never win and +inf costs are comparable: a NaN twist in rollout 0 and beside the
    planted minimum; 1e300 linear velocity (finite force, overflowing square) in every rollout;
    a NaN / +inf mix; an all-NaN batch."""
    L, nr, base = 3, 4099, BIG_BASE
    n = nr * L
    planes, _ = syn.make_planes_torch(n, torch.device("cuda", 0), seed=81)
    v, r22 = planes[0], planes[R22]
    orig, orig_r22 = v.clone(), r22.clone()
    p = 2500
    r22[p * L:(p + 1) * L] = 0.0
    for r in (0, p - 1, p + 1):
        v[r * L + 1] = NAN
    cost, best = _rollout(torch, lib, handle, planes, L, ref=ZERO_W, index_base=base)
    c = cost.cpu().numpy()
    assert np.isnan(c[[0, p - 1, p + 1]]).all() and bits(c[p]) == 0
    assert np.all(np.delete(c, [0, p - 1, p + 1, p]) > 0)
    _assert_best(best, (0.0, p + base), "NaN beside the planted minimum")

    v.copy_(orig)
    r22.copy_(orig_r22)
    v[0::L] = 1e300
    cost, best = _rollout(torch, lib, handle, planes, L, ref=ZERO_W, index_base=base)
    assert bool(torch.isposinf(cost).all()), "1e300 m/s must make every cost +inf"
    _assert_best(best, (INF, base), "all +inf")

    first_inf = 1000
    v[1:first_inf * L:L] = NAN                 # rollouts 0 .. 999 NaN
    v[first_inf * L + 4::2 * L] = NAN          # then every other rollout NaN
    cost, best = _rollout(torch, lib, handle, planes, L, ref=ZERO_W, index_base=base)
    c = cost.cpu().numpy()
    assert np.isnan(c[:first_inf]).all() and np.isposinf(c[first_inf]) and np.isnan(c).sum() > nr // 4
    _assert_best(best, (INF, first_inf + base), "NaN / +inf mix")
    _assert_best(best, expected_best(c, base), "NaN / +inf mix")

    v.fill_(NAN)
    cost, best = _rollout(torch, lib, handle, planes, L, ref=ZERO_W, index_base=base)
    assert bool(torch.isnan(cost).all())
    _assert_best(best, (INF, -1), "all NaN")


def test_empty_batch(torch, lib, handle):
    """n_rollouts = 0: (+inf, -1) and nothing else written."""
    planes = torch.zeros((30, 32), dtype=torch.float64, device="cuda")
    cost = torch.full((4,), SENTINEL, dtype=torch.float64, device="cuda")
    _, best = _rollout(torch, lib, handle, planes, 32, cost_ptr=cost.data_ptr(), n_rollouts=0)
    _assert_best(best, (INF, -1), "empty batch")
    assert bool((cost == SENTINEL).all())


# --- E. windows combined with blf_ccm_argmin_pairs ----------------------------------------------------

def _pairs_tensor(torch, bests):
    return torch.stack([b.cpu() for b in bests]).cuda() if bests else torch.zeros((1, 2), dtype=torch.int64,
                                                                                  device="cuda")


def _argmin_pairs(torch, lib, h, pairs, n=None):
    best = torch.empty(2, dtype=torch.int64, device="cuda")
    rc = lib.blf_ccm_argmin_pairs(h.ptr, pairs.shape[0] if n is None else n, pairs.data_ptr(), best.data_ptr(),
                                  _stream(torch))
    assert rc == 0, lib.blf_ccm_last_error().decode()
    return best


WINDOWS = [(256, (1, 31, 100, 168), True), (3, (32, 96, 4096, 776), True),
           (33, (1, 31, 968, 1000), False), (3, (5, 100, 4000, 895), False)]


@pytest.mark.parametrize("rollout_len,sizes,aligned", WINDOWS, ids=lambda v: str(v))
def test_windows_combined(torch, lib, handle, oracle, rollout_len, sizes, aligned):
    """A batch split into windows (index_base = each window's first rollout), the windows' pairs
    combined with blf_ccm_argmin_pairs; exact ties planted in two windows.  Windows that start on a
    contact index = 0 (mod 32) reproduce the whole call's cost bits and best; others are within
    tolerance and give the selection rule of the concatenated costs."""
    L, nr = rollout_len, sum(sizes)
    st = syn.make_states(nr * L, seed=90 + L, heterogeneous=True)
    starts = np.cumsum((0,) + sizes)
    ties = [int(starts[2]) + 3, int(starts[3]) + 1]
    for r in ties:
        st["poses"][r * L:(r + 1) * L, 11] = 0.0              # R(2,2)
    planes, prm = _states_planes(torch, st)
    whole_cost, whole_best = _rollout(torch, lib, handle, planes, L, prm, ref=ZERO_W)
    bests, costs = [], []
    for a, b in zip(starts[:-1], starts[1:]):
        c, bb = _rollout(torch, lib, handle, planes[:, a * L:b * L], L, prm[:, a * L:b * L], ref=ZERO_W,
                         index_base=int(a))
        bests.append(bb)
        costs.append(c)
    combined = _argmin_pairs(torch, lib, handle, _pairs_tensor(torch, bests))
    cat = torch.cat(costs).cpu().numpy()
    w = oracle.eval_batch_states(st, mask=1, nthreads=8)["wrench"]
    assert_costs_within(cat, oracle.rollout_cost(w, L, ZERO_W, WTS), cost_scale(w, L, ZERO_W, WTS), "windows")
    assert np.all(np.delete(cat, ties) > 0) and all(bits(cat[r]) == 0 for r in ties)
    _assert_best(combined, (0.0, ties[0]), "combined windows")
    _assert_best(combined, expected_best(cat), "combined windows")
    if aligned:
        assert all((int(a) * L) % 32 == 0 for a in starts[:-1])
        assert np.array_equal(cat.view(np.uint64), whole_cost.cpu().numpy().view(np.uint64))
        assert torch.equal(combined, whole_best)


# --- F. blf_ccm_argmin_pairs directly ------------------------------------------------------------------

def _pack(torch, cost, idx):
    p = np.empty((max(1, len(cost)), 2), dtype=np.int64)
    if len(cost):
        p[:, 0] = np.asarray(cost, dtype=np.float64).view(np.int64)
        p[:, 1] = idx
    return _dev(torch, p)


def _check_pairs(torch, lib, h, cost, idx, what):
    best = _argmin_pairs(torch, lib, h, _pack(torch, cost, idx), n=len(cost))
    _assert_best(best, best_of_pairs(cost, idx), what)
    return _decode(best)


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 1000, 4099])
def test_argmin_pairs(torch, lib, handle, n):
    """The minimum at every lane residue and at the last entry; ties and -0.0 against +0.0 (the
    lower index wins with its own bits); NaN never wins; idx -1 / -2 are skipped even with a lower
    cost; (+inf, -1) when every pair is skipped."""
    rng = np.random.default_rng(n)
    h = handle
    idx = rng.permutation(n).astype(np.int64) * 3 + 5          # indices not in position order
    base = rng.uniform(1.0, 2.0, n)
    if n == 0:
        assert _check_pairs(torch, lib, h, [], [], "n=0")[1] == -1
        return
    sites = sorted({min(n - 1, r + 32 * int(rng.integers(0, max(1, n // 32)))) for r in range(min(n, 32))} | {n - 1})
    for j in sites:
        c = base.copy()
        c[j] = 0.5
        assert _check_pairs(torch, lib, h, c, idx, f"n={n} min at {j}")[1] == idx[j]
        if n > 1:                                              # an exact tie elsewhere
            k = (j + 1 + int(rng.integers(0, n - 1))) % n
            c[k] = 0.5
            _check_pairs(torch, lib, h, c, idx, f"n={n} tie {j}/{k}")
            c[j], c[k] = -0.0, 0.0                              # -0.0 == +0.0: the lower index wins
            got = _check_pairs(torch, lib, h, c, idx, f"n={n} -0.0 at {j}, +0.0 at {k}")
            assert got[1] == min(idx[j], idx[k])
            c[j], c[k] = 0.0, -0.0
            _check_pairs(torch, lib, h, c, idx, f"n={n} +0.0 at {j}, -0.0 at {k}")
    c = base.copy()
    c[rng.random(n) < 0.5] = NAN
    c[0] = NAN
    _check_pairs(torch, lib, h, c, idx, f"n={n} NaNs")
    skip = idx.copy()
    neg = rng.random(n) < 0.3
    neg[0] = neg[-1] = True
    skip[neg] = np.where(rng.random(int(neg.sum())) < 0.5, -1, -2)
    c = base.copy()
    c[neg] = -5.0                                              # lower, but skipped
    got = _check_pairs(torch, lib, h, c, skip, f"n={n} negative indices")
    assert got[1] >= 0 or neg.all()
    _check_pairs(torch, lib, h, base, np.full(n, -1), f"n={n} every pair skipped")
    _check_pairs(torch, lib, h, np.full(n, NAN), idx, f"n={n} all NaN")
    _check_pairs(torch, lib, h, np.full(n, INF), idx, f"n={n} all +inf")


# --- G. scratch growth, guard bands, determinism ------------------------------------------------------

GUARD = 37


def test_scratch_growth_guards_and_determinism(torch, lib, handle):
    """small -> large (the handle's partials are reallocated) -> small on one handle, each bit for
    bit a fresh handle's result; cost and a 16-byte best inside sentinel guard bands; a repeated
    call gives the same bits."""
    shapes = [(33, 40, 11), (256, 4099, 12), (33, 40, 11), (1, 5000, 13)]
    h = _new_handle()
    try:
        for L, nr, seed in shapes:
            st = syn.make_states(nr * L, seed=seed, heterogeneous=True)
            planes, prm = _states_planes(torch, st)
            cbuf = torch.full((nr + 2 * GUARD,), SENTINEL, dtype=torch.float64, device="cuda")
            bbuf = torch.full((10,), -77, dtype=torch.int64, device="cuda")
            cost_v, best_v = cbuf[GUARD:GUARD + nr], bbuf[4:6]
            assert best_v.data_ptr() % 16 == 0
            _rollout(torch, lib, h, planes, L, prm, index_base=BIG_BASE, cost_ptr=cost_v.data_ptr(),
                     best_ptr=best_v.data_ptr())
            what = f"L={L} n_rollouts={nr}"
            assert bool((cbuf[:GUARD] == SENTINEL).all()) and bool((cbuf[GUARD + nr:] == SENTINEL).all()), \
                f"{what}: cost guard band written"
            rest = torch.cat([bbuf[:4], bbuf[6:]])
            assert bool((rest == -77).all()), f"{what}: best guard band written"
            c = cost_v.cpu().numpy()
            assert np.all(np.isfinite(c))
            _assert_best(best_v, expected_best(c, BIG_BASE), what)
            again_c, again_b = _rollout(torch, lib, h, planes, L, prm, index_base=BIG_BASE)
            assert torch.equal(again_c, cost_v) and torch.equal(again_b, best_v), f"{what}: not deterministic"
            fresh = _new_handle()
            try:
                fc, fb = _rollout(torch, lib, fresh, planes, L, prm, index_base=BIG_BASE)
                torch.cuda.synchronize()
            finally:
                fresh.close()
            assert torch.equal(fc, cost_v) and torch.equal(fb, best_v), f"{what}: differs from a fresh handle"
    finally:
        h.close()


# --- H. the reduction fed by the fused rollout ----------------------------------------------------------

@pytest.mark.parametrize("ws", ["3", None], ids=["ws2-form", "default-form"])
def test_fused_rollout_reduction_past_one_pass(torch, lib, monkeypatch, ws):
    """blf_ccm_rollout_integrate_cost with 2^20 + 33 one-foot, one-step rollouts: its two-launch forms
    feed ccm_cost_reduce_kernel with fixed_count.  Chains with spring = damper = 0 cost exactly
    +0.0; the lowest planted one wins against ties in the other pass."""
    if ws is None:
        monkeypatch.delenv("BLF_CCM_TUNE_ROLLOUT_WS", raising=False)
    else:
        monkeypatch.setenv("BLF_CCM_TUNE_ROLLOUT_WS", ws)
    h = _new_handle()
    try:
        nr = PASS + 33
        planes, prm = syn.make_planes_torch(nr, torch.device("cuda", 0), seed=97, heterogeneous=True)
        tw, pos, rot, nul = planes[0:6], planes[6:9], planes[9:18], planes[18:30]
        best = torch.empty(2, dtype=torch.int64, device="cuda")
        cost = torch.empty(nr, dtype=torch.float64, device="cuda")
        ref, wts = np.ascontiguousarray(ZERO_W), np.ascontiguousarray(WTS)
        sites = [0, 127, PASS - 1, PASS, PASS + 1, nr - 1]
        for r in sites:
            prm[2][r] = 0.0
            prm[3][r] = 0.0
        for k, lowest in enumerate(sites):
            before = h.launch_count
            rc = lib.blf_ccm_rollout_integrate_cost(
                h.ptr, nr, 1, 1, 0.01, 0.0, _pp(tw, 6), _pp(pos, 3), _pp(rot, 9), _pp(nul, 12), _pp(prm, 4), 0,
                None, None, None, None, None, ref.ctypes.data, wts.ctypes.data, 5, cost.data_ptr(),
                best.data_ptr(), _stream(torch))
            assert rc == 0, lib.blf_ccm_last_error().decode()
            assert h.launch_count - before == 2                # rollout kernel + ccm_cost_reduce_kernel
            what = f"BLF_CCM_TUNE_ROLLOUT_WS={ws} planted {sites[k:]}"
            _check_planted(torch, cost, sites[k:], what)
            _assert_best(best, (0.0, lowest + 5), what)
            prm[2][lowest] = 1.0e4
            prm[3][lowest] = 1.0e2
    finally:
        h.close()
