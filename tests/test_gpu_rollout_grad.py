"""GPU tests of the rollout cost's reverse mode (blf_ccm_rollout_cost_vjp, RolloutBatch.cost_vjp /
prepare_cost_vjp / rollout_cost, the C++ rolloutCostGradient): against 80-digit forward mode and
central differences (tests/golden/rollout_grad_golden.npz) and the float64 torch restatement of
tests/rollout_grad_reference.py, bit for bit against blf_ccm_wrench_vjp_soa at H = 1, every
gradient-group subset, argument checks, guard bands, determinism and torch.autograd."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rollout_grad_reference as ref
from test_rollout_grad_oracle import WORST_F64
from bipedal_locomotion_framework_b200 import _capi

pytestmark = pytest.mark.gpu

TOL_SHORT = 1e-12
TOL_LONG = 1000 * WORST_F64[100]   # 1e-12: float64 reaches 1e-15 against the 80-digit differences
NAMES = ("twist", "pos", "rot", "null", "params")
ROWS = {"twist": 6, "pos": 3, "rot": 9, "null": 12, "params": 4}
SENTINEL = -123.25


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need the B200"
    return torch


@pytest.fixture(scope="module")
def rb(torch):
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    from bipedal_locomotion_framework_b200.system import RolloutBatch
    return RolloutBatch(ContinuousContactModelBatch(0))


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _inputs(torch, rb, case):
    """Device planes of a case; uniform parameters go to the handle (param_planes None)."""
    d = {k: _dev(torch, case[k]) for k in ("twist", "pos", "rot", "null")}
    if case["het"]:
        d["params"] = _dev(torch, case["params"])
    else:
        rb._b.set_uniform_params(*case["uniform"])
        d["params"] = None
    return d


def _args(case, dT, rho, d):
    return (case["n_rollouts"], case["feet"], case["horizon"], dT, rho, d["twist"], d["pos"], d["rot"],
            d["null"], ref.REF, ref.WEIGHTS)


def _vjp(torch, rb, case, dT, rho, inputs=True, gcost=None):
    d = _inputs(torch, rb, case)
    g = _dev(torch, case["grad_cost"] if gcost is None else gcost)
    out = rb.cost_vjp(*_args(case, dT, rho, d), g, param_planes=d["params"], inputs=inputs)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("row", ref.SHORT_CASES, ids=[r[0] for r in ref.SHORT_CASES])
def test_against_forward_mode(torch, rb, row):
    case, dT, rho = ref.case_from_row(row)
    got = _vjp(torch, rb, case, dT, rho)
    dual = ref.load_golden()[row[0] + "/dual"]
    for c in range(case["n_rollouts"] * case["feet"]):
        v = ref.chain_vector(got, case, c) / case["grad_cost"][c // case["feet"]]
        err = ref.group_errors(v, dual[c], case["horizon"])
        assert max(err.values()) <= TOL_SHORT, (row[0], c, err)


@pytest.mark.parametrize("row", ref.LONG_CASES, ids=[r[0] for r in ref.LONG_CASES])
def test_against_central_differences(torch, rb, row):
    case, dT, rho = ref.case_from_row(row)
    got = _vjp(torch, rb, case, dT, rho)
    gd = ref.load_golden()
    for c in range(case["n_rollouts"] * case["feet"]):
        v = ref.chain_vector(got, case, c) / case["grad_cost"][c // case["feet"]]
        err = np.max(np.abs(v[gd[row[0] + "/coords"][c]] - gd[row[0] + "/fd"][c])) / np.linalg.norm(v)
        assert err <= TOL_LONG, (row[0], c, err)


def _torch_check(torch, rb, case, dT, rho, tol):
    got = _vjp(torch, rb, case, dT, rho)
    want, _ = ref.torch_grads(case, dT, rho)
    H, chains = case["horizon"], case["n_rollouts"] * case["feet"]
    worst = 0.0
    for c in range(chains):
        err = ref.group_errors(ref.chain_vector(got, case, c), ref.chain_vector(want, case, c), H)
        worst = max(worst, *err.values())
    assert worst <= tol, worst
    return got


@pytest.mark.parametrize("n_rollouts,feet,horizon,rho,het", [
    (4096, 2, 100, 0.01, False),   # the MPC size
    (4096, 2, 100, 0.0, True),
    (499, 3, 37, 0.02, True),      # ragged: 1 497 chains, 37 steps
])
def test_against_torch_restatement(torch, rb, n_rollouts, feet, horizon, rho, het):
    case = ref.make_case(n_rollouts, feet, horizon, seed=n_rollouts + horizon, het=het, inverted=True, at_null=True)
    _torch_check(torch, rb, case, 0.01, rho, TOL_LONG)


@pytest.mark.parametrize("feet", [1, 2, 4])
@pytest.mark.parametrize("horizon", [1, 2, 7, 8, 9, 15, 16, 17, 23])
def test_feet_and_horizons(torch, rb, feet, horizon):
    case = ref.make_case(24 // feet + 1, feet, horizon, seed=7 * feet + horizon, het=feet == 2, inverted=True)
    _torch_check(torch, rb, case, 0.01, 0.3, TOL_SHORT if horizon <= 6 else TOL_LONG)


def _close(got, want, tol, what):
    """Norm-wise per (chain, plane group): |got - want| / |want| <= tol (absolute where want is zero)."""
    got, want = np.asarray(got).reshape(got.shape[0], -1), np.asarray(want).reshape(want.shape[0], -1)
    num = np.linalg.norm(got - want, axis=0)
    den = np.linalg.norm(want, axis=0)
    err = num / np.where(den > 0, den, 1.0)
    assert err.max() <= tol, (what, err.max())


# nvcc contracts the products of the shared closed forms (eval_contact, vjp_wrench) into FMAs
# differently in different kernels (as between ccm_single_kernel and ccm_aos_kernel), so these
# comparisons hold to a few ulp of each block, not bit for bit.
TOL_ULP = 1e-14


@pytest.mark.parametrize("het", [False, True])
@pytest.mark.parametrize("rho", [0.0, 0.4])
def test_horizon_one_equals_the_wrench_vjp(torch, rb, het, rho):
    case = ref.make_case(40, 2, 1, seed=99, het=het, inverted=True, at_null=True)
    case["rot"][:, 2] = (np.diag([1.0, 1.0, 0.0]) @ np.eye(3)).reshape(9)     # R22 = +0
    d = _inputs(torch, rb, case)
    fwd = rb.run(*_args(case, 0.01, rho, d), param_planes=d["params"], mask=_capi.WRENCH)
    gcost = _dev(torch, case["grad_cost"])
    got = rb.cost_vjp(*_args(case, 0.01, rho, d), gcost, param_planes=d["params"])
    gbar = gcost.repeat_interleave(2)
    F, Ref = fwd["wrench"], torch.tensor(ref.REF, device="cuda")[:, None]
    w = torch.tensor([ref.WEIGHTS[0]] * 3 + [ref.WEIGHTS[1]] * 3, device="cuda")[:, None]
    cot = (2.0 * gbar[None, :] * w) * (F - Ref)
    planes = torch.cat([d["twist"], d["pos"], d["rot"], d["null"]]).contiguous()
    prm = d["params"] if het else None
    want = rb._b.wrench_vjp(planes, cot.contiguous(), prm, params=True)
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy() for k, v in got.items()}
    wp, wq = want["planes"].cpu().numpy(), want["params"].cpu().numpy()
    blocks = {"v": (got["twist"][0:3], wp[0:3]), "w": (got["twist"][3:6], wp[3:6]),
              "p": (got["pos"], wp[6:9]), "R": (got["rot"], wp[9:18]), "p0": (got["null"][0:3], wp[18:21]),
              "R0": (got["null"][3:], wp[21:30]), "params": (got["params"], wq)}
    for name, (g, x) in blocks.items():
        _close(g, x, TOL_ULP, name)
    # the structurally dead entries are +0.0 in both
    for g in (got["rot"][[2, 5]], got["null"][[5, 8, 11]]):
        assert (g == 0.0).all() and not np.signbit(g).any()
    r22 = case["rot"][8] == 0.0
    assert r22.any() and (got["rot"][8][r22] == wp[17][r22]).all()   # sgn(+-0) = 0 in both


def test_every_group_subset(torch, rb):
    case = ref.make_case(37, 2, 13, seed=5, het=True, inverted=True)
    full = _vjp(torch, rb, case, 0.01, 0.2)
    groups = ["twist", "pose", "null", "params"]
    for mask in range(1, 16):
        sub = {g for i, g in enumerate(groups) if mask >> i & 1}
        got = _vjp(torch, rb, case, 0.01, 0.2, inputs=sub)
        keys = {k for g in sub for k in (("pos", "rot") if g == "pose" else (g,))}
        assert set(got) == keys, mask
        for k in keys:
            _close(got[k], full[k], TOL_ULP, (mask, k))


def _raw_call(torch, rb, case, d, gcost, outs, n_rollouts=None, feet=None, horizon=None, **over):
    pp = lambda t, cnt: None if t is None else _capi_ptrs(t, cnt)
    args = dict(tw=pp(d["twist"], 6), pos=pp(d["pos"], 3), rot=pp(d["rot"], 9), null=pp(d["null"], 12),
                prm=pp(d["params"], 4), gcost=None if gcost is None else gcost.data_ptr(),
                gtw=pp(outs.get("twist"), 6), gpos=pp(outs.get("pos"), 3), grot=pp(outs.get("rot"), 9),
                gnul=pp(outs.get("null"), 12), gprm=pp(outs.get("params"), 4))
    args.update(over)
    ref_ = np.array(ref.REF)
    wts = np.array(ref.WEIGHTS)
    return _capi.lib().blf_ccm_rollout_cost_vjp(
        rb._b.handle.ptr, case["n_rollouts"] if n_rollouts is None else n_rollouts,
        case["feet"] if feet is None else feet, case["horizon"] if horizon is None else horizon, 0.01, 0.2,
        args["tw"], args["pos"], args["rot"], args["null"], args["prm"], ref_.ctypes.data, wts.ctypes.data,
        args["gcost"], args["gtw"], args["gpos"], args["grot"], args["gnul"], args["gprm"], None)


def _capi_ptrs(t, cnt):
    if isinstance(t, list):
        return (C.c_void_p * cnt)(*[None if p is None else (p if isinstance(p, int) else p.data_ptr()) for p in t])
    return (C.c_void_p * cnt)(*[t[i].data_ptr() for i in range(cnt)])


def test_argument_checks_launch_nothing(torch, rb):
    case = ref.make_case(5, 2, 9, seed=3, het=True)
    d = _inputs(torch, rb, case)
    gcost = _dev(torch, case["grad_cost"])
    chains = 10
    mk = lambda r, n: torch.zeros((r, n), dtype=torch.float64, device="cuda")
    outs = {"twist": mk(6, 9 * chains), "pos": mk(3, chains), "rot": mk(9, chains), "null": mk(12, chains),
            "params": mk(4, chains)}
    L = _capi.lib()
    h = rb._b.handle
    assert _raw_call(torch, rb, case, d, gcost, outs) == 0, L.blf_ccm_last_error()
    torch.cuda.synchronize()
    before = h.launch_count
    E = _capi.ERR_INVALID_ARG
    assert _raw_call(torch, rb, case, d, gcost, {}) == E                            # nothing requested
    assert _raw_call(torch, rb, case, d, None, outs) == E                           # grad_cost NULL
    assert _raw_call(torch, rb, case, d, gcost, outs, n_rollouts=0) == 0            # no-op
    assert _raw_call(torch, rb, case, d, gcost, outs, n_rollouts=0, feet=0) == 0
    assert _raw_call(torch, rb, case, d, gcost, outs, feet=0) == E
    assert _raw_call(torch, rb, case, d, gcost, outs, horizon=0) == E
    assert _raw_call(torch, rb, case, d, gcost, {"pos": outs["pos"]}) == E          # pos without rot
    for key, cnt, src in (("tw", 6, d["twist"]), ("pos", 3, d["pos"]), ("rot", 9, d["rot"]),
                          ("null", 12, d["null"]), ("prm", 4, d["params"]), ("gtw", 6, outs["twist"]),
                          ("gpos", 3, outs["pos"]), ("grot", 9, outs["rot"]), ("gnul", 12, outs["null"]),
                          ("gprm", 4, outs["params"])):
        for i in range(cnt):
            if key == "null" and i in (5, 8, 11):
                continue
            for bad in (None, src[i].data_ptr() + 4):
                planes = [src[j] for j in range(cnt)]
                planes[i] = bad
                assert _raw_call(torch, rb, case, d, gcost, outs, **{key: _capi_ptrs(planes, cnt)}) == E, (key, i)
    assert h.launch_count == before
    # the null pose's third rotation column is never read
    planes = [d["null"][j] for j in range(12)]
    for j in (5, 8, 11):
        planes[j] = None
    assert _raw_call(torch, rb, case, d, gcost, outs, null=_capi_ptrs(planes, 12)) == 0
    # no parameters at all
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    from bipedal_locomotion_framework_b200.system import RolloutBatch
    fresh = RolloutBatch(ContinuousContactModelBatch(0))
    d2 = dict(d, params=None)
    assert _raw_call(torch, fresh, case, d2, gcost, outs) == _capi.ERR_NOT_INITIALIZED


def test_guard_bands_and_dead_planes(torch, rb):
    case = ref.make_case(21, 2, 11, seed=8, het=True, inverted=True)
    full = _vjp(torch, rb, case, 0.01, 0.2)
    d = _inputs(torch, rb, case)
    chains, G = 42, 64
    outs, bufs = {}, {}
    for k, rows in ROWS.items():
        n = 11 * chains if k == "twist" else chains
        bufs[k] = torch.full((rows, n + 2 * G), SENTINEL, dtype=torch.float64, device="cuda")
        outs[k] = [bufs[k][i, G:G + n] for i in range(rows)]
    assert _raw_call(torch, rb, case, d, _dev(torch, case["grad_cost"]), outs) == 0
    torch.cuda.synchronize()
    for k in ROWS:
        b = bufs[k].cpu().numpy()
        assert (b[:, :G] == SENTINEL).all() and (b[:, -G:] == SENTINEL).all(), k
        assert np.array_equal(b[:, G:-G], full[k]), k
    assert (full["null"][[5, 8, 11]] == 0.0).all() and not np.signbit(full["null"][[5, 8, 11]]).any()


def test_repeated_runs_are_bit_identical_and_prepared_form_matches(torch, rb):
    case = ref.make_case(300, 2, 50, seed=12, het=False, inverted=True)
    a = _vjp(torch, rb, case, 0.01, 0.05)
    b = _vjp(torch, rb, case, 0.01, 0.05)
    d = _inputs(torch, rb, case)
    call, out = rb.prepare_cost_vjp(*_args(case, 0.01, 0.05, d), _dev(torch, case["grad_cost"]))
    call()
    call()
    torch.cuda.synchronize()
    for k in a:
        assert np.array_equal(a[k].view(np.int64), b[k].view(np.int64)), k
        assert np.array_equal(a[k].view(np.int64), out[k].cpu().numpy().view(np.int64)), k


def test_autograd_gradcheck(torch, rb):
    case = ref.make_case(2, 2, 3, seed=4, het=True, inverted=True)
    d = {k: _dev(torch, case[k]).requires_grad_() for k in NAMES}
    fn = lambda tw, p, r, n, q: rb.rollout_cost(2, 2, 3, 0.01, 0.3, tw, p, r, n, ref.REF, [1e-6, 1e-5], q)
    assert torch.autograd.gradcheck(fn, tuple(d[k] for k in NAMES), eps=1e-7, atol=1e-6, rtol=1e-5)


def test_autograd_asks_only_for_needed_groups(torch, rb, monkeypatch):
    case = ref.make_case(3, 2, 4, seed=6)
    seen = []
    real = rb.cost_vjp
    monkeypatch.setattr(rb, "cost_vjp", lambda *a, **k: seen.append(k["inputs"]) or real(*a, **k))
    rb._b.set_uniform_params(*case["uniform"])
    tw = _dev(torch, case["twist"]).requires_grad_()
    cost = rb.rollout_cost(3, 2, 4, 0.01, 0.1, tw, _dev(torch, case["pos"]), _dev(torch, case["rot"]),
                           _dev(torch, case["null"]), ref.REF, ref.WEIGHTS)
    cost.sum().backward()
    assert seen == [{"twist"}]
    want, _ = ref.torch_grads(case, 0.01, 0.1, grad_cost=np.ones(3))
    np.testing.assert_allclose(tw.grad.cpu().numpy(), want["twist"], rtol=1e-11, atol=1e-11 * np.abs(want["twist"]).max())


def test_gradient_step_lowers_the_cost(torch, rb):
    case = ref.make_case(256, 2, 100, seed=21, het=True)
    d = _inputs(torch, rb, case)
    tw = d["twist"].clone().requires_grad_()
    cost = rb.rollout_cost(*_args(case, 0.01, 0.02, dict(d, twist=tw)), param_planes=d["params"])
    cost.sum().backward()
    g = tw.grad
    step = 1e-3 * cost.sum() / (g * g).sum()
    after = rb.run(*_args(case, 0.01, 0.02, dict(d, twist=(tw - step * g).detach())), param_planes=d["params"])["cost"]
    assert float(after.sum()) < float(cost.detach().sum()) * (1 - 1e-4)
    assert bool((after <= cost.detach() * (1 + 1e-12)).float().mean() > 0.9)


def test_cpp_rollout_gradient_executable(torch):
    from bipedal_locomotion_framework_b200 import build as b
    exe = os.path.join(b.LIB_DIR, "RolloutGradientUnitTests")
    assert os.path.exists(exe), "build() builds the C++ test executables"
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0, r.stdout
