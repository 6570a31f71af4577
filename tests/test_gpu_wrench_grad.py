"""GPU tests of the wrench's reverse mode (blf_ccm_wrench_vjp_soa, ContinuousContactModelBatch.
wrench_vjp / contact_wrench, the C++ wrenchGradient): against the exact Jacobians and the torch
restatement of tests/wrench_grad_reference.py at 1e-12 per block (scale: the larger of the block's
norm and its operand magnitude), every gradient-group subset, memory safety, consistency with the
forward pass and the control matrix, and torch.autograd."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import wrench_grad_reference as ref
from bipedal_locomotion_framework_b200 import _capi
from bipedal_locomotion_framework_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

TOL = 1e-12
GROUP_NAMES = ("twist", "pose", "null_pose")
GROUP_ROWS = {"twist": range(0, 6), "pose": range(6, 18), "null_pose": range(18, 30)}
SENTINEL = -123.25


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


def _dev(torch, a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _states(n, seed, het):
    st = syn.make_states(max(n, 1), seed=seed, heterogeneous=het)
    planes = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])[:, :n]
    prm = st["params"].T[:, :n] if het else np.tile(np.array(syn.REFERENCE_TEST_PARAMS)[:, None], (1, n))
    return np.ascontiguousarray(planes), np.ascontiguousarray(prm)


def _check(got_x, got_p, planes, prm, g, what, want=None):
    want_x, want_p = want if want is not None else ref.torch_vjp(planes, prm, g)
    mag_x, mag_p = ref.operand_magnitude(planes, prm, g)
    err = ref.vjp_errors(got_x, got_p, want_x, want_p, mag_x, mag_p)
    if err is not None and err.size:
        i = int(err.argmax())
        assert err[i] <= TOL, f"{what}: contact {i} rel err {err[i]:.3e}"
    if got_x is not None:
        assert np.all(got_x[list(ref.DEAD_PLANES)] == 0.0) and not np.signbit(got_x[list(ref.DEAD_PLANES)]).any()


# --- parity with the references ---------------------------------------------------------------------

def test_exact_golden_jacobians(torch, batch):
    gd = ref.load_golden()
    planes, prm = ref.golden_planes(gd)
    n = planes.shape[1]
    rng = np.random.default_rng(11)
    for trial in range(7):
        g = np.zeros((6, n))
        if trial < 6:
            g[trial] = 1.0
        else:
            g = rng.uniform(-1, 1, (6, n))
        out = batch.wrench_vjp(_dev(torch, planes), _dev(torch, g), _dev(torch, prm), params=True)
        _check(out["planes"].cpu().numpy(), out["params"].cpu().numpy(), planes, prm, g,
               f"golden/cotangent {trial}", want=ref.golden_vjp(gd, g))


@pytest.mark.parametrize("het", [False, True])
def test_seeded_batch_against_the_torch_restatement(torch, batch, het):
    n = 819200
    planes, prm = _states(n, 42 + 7 * het, het)
    g = np.random.default_rng(het).uniform(-1, 1, (6, n)) * np.array([1, 1, 1, 10, 10, 10])[:, None]
    out = batch.wrench_vjp(_dev(torch, planes), _dev(torch, g), _dev(torch, prm) if het else None,
                           params=True)
    _check(out["planes"].cpu().numpy(), out["params"].cpu().numpy(), planes, prm, g, f"het={het}")


@pytest.mark.parametrize("n", [0, 1, 31, 32, 33, 63, 65, 129, 4097])
def test_ragged_sizes(torch, batch, n):
    planes, prm = _states(n, 5, True)
    g = np.random.default_rng(n).uniform(-1, 1, (6, n))
    launches = batch.handle.launch_count
    out = batch.wrench_vjp(_dev(torch, planes), _dev(torch, g), _dev(torch, prm), params=True)
    assert batch.handle.launch_count == launches + (1 if n else 0)
    if n:
        _check(out["planes"].cpu().numpy(), out["params"].cpu().numpy(), planes, prm, g, f"n={n}")


# --- group subsets, dead planes, argument errors ---------------------------------------------------------

def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])


@pytest.mark.parametrize("groups", list(range(1, 16)))
def test_every_group_subset(torch, batch, groups):
    n = 777
    planes, prm = _states(n, 9, True)
    g = np.random.default_rng(groups).uniform(-1, 1, (6, n))
    want_x, want_p = ref.torch_vjp(planes, prm, g)
    names = [nm for b, nm in enumerate(GROUP_NAMES) if groups & (1 << b)]
    want_params = bool(groups & 8)
    # planes no requested gradient reads are passed as NULL
    read = set(ref.LIVE_PLANES) if ({"pose"} & set(names) or want_params) else {9, 10, 12, 13, 15, 16, 17}
    dp, dprm, dg = _dev(torch, planes), _dev(torch, prm), _dev(torch, g)
    inp = [dp[i] if i in read else None for i in range(30)]
    gx = torch.full((30, n), SENTINEL, dtype=torch.float64, device="cuda")
    gp = torch.full((4, n), SENTINEL, dtype=torch.float64, device="cuda")
    rows = {i for nm in names for i in GROUP_ROWS[nm]}
    rc = _capi.lib().blf_ccm_wrench_vjp_soa(
        batch.handle.ptr, n, _ptrs(inp), _ptrs(list(dprm)), _ptrs(list(dg)),
        _ptrs([gx[i] if i in rows else None for i in range(30)]) if rows else None,
        _ptrs(list(gp)) if want_params else None, None)
    assert rc == 0, _capi.lib().blf_ccm_last_error()
    got_x, got_p = gx.cpu().numpy(), gp.cpu().numpy()
    for i in range(30):
        if i not in rows:
            assert np.all(got_x[i] == SENTINEL), i
    if not want_params:
        assert np.all(got_p == SENTINEL)
    sel = np.array(sorted(rows), dtype=int)
    cx = np.zeros_like(got_x)
    cx[sel] = got_x[sel]
    wx = np.zeros_like(want_x)
    wx[sel] = want_x[sel]
    _check(cx if rows else None, got_p if want_params else None, planes, prm, g, f"groups={groups}",
           want=(wx, want_p))
    # a plane a requested gradient reads may not be NULL
    need = sorted(read)[0]
    bad = list(inp)
    bad[need] = None
    rc = _capi.lib().blf_ccm_wrench_vjp_soa(
        batch.handle.ptr, n, _ptrs(bad), _ptrs(list(dprm)), _ptrs(list(dg)),
        _ptrs([gx[i] if i in rows else None for i in range(30)]) if rows else None,
        _ptrs(list(gp)) if want_params else None, None)
    assert rc == _capi.ERR_INVALID_ARG


def test_argument_errors_and_null_cotangents(torch, batch):
    L = _capi.lib()
    n = 100
    planes, prm = _states(n, 3, False)
    dp = _dev(torch, planes)
    g = np.random.default_rng(0).uniform(-1, 1, (6, n))
    g[1] = 0.0
    g[4] = 0.0
    dg = _dev(torch, g)
    gx = torch.empty((30, n), dtype=torch.float64, device="cuda")
    args = lambda m, gw, gin: (batch.handle.ptr, m, _ptrs(list(dp)), None, gw, gin, None, None)
    assert L.blf_ccm_wrench_vjp_soa(*args(-1, _ptrs(list(dg)), _ptrs(list(gx)))) == _capi.ERR_INVALID_ARG
    assert L.blf_ccm_wrench_vjp_soa(*args(n, _ptrs(list(dg)), None)) == _capi.ERR_INVALID_ARG
    assert L.blf_ccm_wrench_vjp_soa(None, n, None, None, None, None, None, None) == _capi.ERR_INVALID_HANDLE
    launches = batch.handle.launch_count
    assert L.blf_ccm_wrench_vjp_soa(*args(0, _ptrs(list(dg)), _ptrs(list(gx)))) == 0
    assert batch.handle.launch_count == launches
    # NULL cotangent entries count as zero
    gw = [dg[j] if j not in (1, 4) else None for j in range(6)]
    assert L.blf_ccm_wrench_vjp_soa(*args(n, _ptrs(gw), _ptrs(list(gx)))) == 0, L.blf_ccm_last_error()
    _check(gx.cpu().numpy(), None, planes, prm, g, "null cotangents")
    # no cotangent at all: every gradient is zero
    assert L.blf_ccm_wrench_vjp_soa(*args(n, None, _ptrs(list(gx)))) == 0
    assert torch.count_nonzero(gx).item() == 0


# --- memory safety ---------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 33, 4097])
def test_guard_bands_and_eight_byte_aligned_views(torch, batch, n):
    planes, prm = _states(n, 17, True)
    g = np.random.default_rng(n).uniform(-1, 1, (6, n))
    aligned = batch.wrench_vjp(_dev(torch, planes), _dev(torch, g), _dev(torch, prm), params=True)
    guard = 40

    def shifted(a):  # rows start 8- but not 16-byte aligned
        big = torch.empty((a.shape[0], a.shape[1] + 2), dtype=torch.float64, device="cuda")
        v = big[:, 1:a.shape[1] + 1]
        v.copy_(_dev(torch, a))
        assert v[0].data_ptr() % 16 == 8
        return v

    bx = torch.full((30, n + 2 * guard + 1), SENTINEL, dtype=torch.float64, device="cuda")
    bp = torch.full((4, n + 2 * guard + 1), SENTINEL, dtype=torch.float64, device="cuda")
    out = {"planes": bx[:, guard + 1:guard + 1 + n], "params": bp[:, guard + 1:guard + 1 + n]}
    assert out["planes"][0].data_ptr() % 16 == 8
    batch.wrench_vjp(shifted(planes), shifted(g), shifted(prm), params=True, out=out)
    for buf in (bx, bp):
        h = buf.cpu().numpy()
        assert np.all(h[:, :guard + 1] == SENTINEL) and np.all(h[:, guard + 1 + n:] == SENTINEL)
    assert torch.equal(out["planes"], aligned["planes"]) and torch.equal(out["params"], aligned["params"])


# --- consistency with the forward pass and the control matrix ------------------------------------------

def test_jacobian_matches_finite_differences_and_the_control_matrix(torch, batch):
    n = 2048
    planes, prm = _states(n, 23, True)
    dp, dprm = _dev(torch, planes), _dev(torch, prm)
    jac = np.empty((n, 6, ref.NCOLS))
    for r in range(6):
        g = np.zeros((6, n))
        g[r] = 1.0
        out = batch.wrench_vjp(dp, _dev(torch, g), dprm, params=True)
        jac[:, r, :len(ref.LIVE_PLANES)] = out["planes"].cpu().numpy()[ref.LIVE_PLANES].T
        jac[:, r, len(ref.LIVE_PLANES):] = out["params"].cpu().numpy().T

    def wrench(x, q):
        return batch.evaluate_soa(_dev(torch, x), _dev(torch, q), 1)["wrench"].cpu().numpy()

    fd = np.empty_like(jac)
    for c in range(ref.NCOLS):
        x, q = planes.copy(), prm.copy()
        arr, row = (x, ref.LIVE_PLANES[c]) if c < len(ref.LIVE_PLANES) else (q, c - len(ref.LIVE_PLANES))
        h = 1e-6 * np.maximum(1.0, np.abs(arr[row]))
        base = arr[row].copy()
        arr[row] = base + h
        up = wrench(x, q)
        arr[row] = base - h
        dn = wrench(x, q)
        fd[:, :, c] = ((up - dn) / (2 * h)).T
    # the |R22| kink: central differences straddling R22 = 0 are not derivatives
    ok = np.abs(planes[17]) > 1e-4
    scale = np.maximum(np.abs(jac).max(axis=2, keepdims=True), 1e-300)
    err = np.abs(jac - fd) / scale
    print(f"worst central-difference mismatch {err[ok].max():.2e}")
    assert err[ok].max() <= 1e-5, err[ok].max()

    # where R22 > 0: dF/dv and dT/dw are the control matrix's diagonal blocks
    ctrl = batch.evaluate_soa(dp, dprm, 4)["ctrl"].cpu().numpy().reshape(n, 6, 6)
    pos = planes[17] > 0
    cv = [ref.LIVE_PLANES.index(i) for i in range(3)]
    cw = [ref.LIVE_PLANES.index(i) for i in range(3, 6)]
    for blk, cols in ((slice(0, 3), cv), (slice(3, 6), cw)):
        a = jac[pos][:, blk][:, :, cols]
        b = ctrl[pos][:, blk, blk]
        den = np.maximum(np.abs(b).max(axis=(1, 2)), 1e-300)
        assert (np.abs(a - b).max(axis=(1, 2)) / den).max() <= TOL


# --- torch.autograd ---------------------------------------------------------------------------------

def test_gradcheck(torch, batch):
    n = 6
    planes, prm = _states(n, 31, True)
    planes[17] = np.where(np.abs(planes[17]) < 0.05, 0.5, planes[17])   # away from the |R22| kink
    prm[2] = 2000.0 * (1 + np.arange(n))   # moderate stiffness: finite differences stay accurate
    prm[3] = 100.0
    x = _dev(torch, planes).requires_grad_()
    q = _dev(torch, prm).requires_grad_()
    assert torch.autograd.gradcheck(lambda a, b: batch.contact_wrench(a, b), (x, q))


def test_loss_gradients_match_the_cpu_restatement(torch, batch, monkeypatch):
    n = 50000
    planes, prm = _states(n, 37, True)
    target = np.random.default_rng(1).uniform(-5, 5, (6, n))
    wts = torch.tensor([1.0, 1.0, 1.0, 10.0, 10.0, 10.0], dtype=torch.float64, device="cuda")[:, None]

    def loss_fn(w, tgt):
        return (wts.to(w.device) * (w - tgt) ** 2).sum()

    x = _dev(torch, planes).requires_grad_()
    q = _dev(torch, prm).requires_grad_()
    w = batch.contact_wrench(x, q)
    loss_fn(w, _dev(torch, target)).backward()
    xc = torch.from_numpy(planes).requires_grad_()
    qc = torch.from_numpy(prm).requires_grad_()
    wc = ref.torch_wrench(xc, qc)
    loss_fn(wc, torch.from_numpy(target)).backward()
    gbar = (2 * wts.cpu() * (wc.detach() - torch.from_numpy(target))).numpy()
    _check(x.grad.cpu().numpy(), q.grad.cpu().numpy(), planes, prm, gbar, "loss",
           want=(xc.grad.numpy(), qc.grad.numpy()))

    # only the state requires grad: the backward asks for no parameter group
    calls = []
    real = batch.wrench_vjp

    def spy(*a, **k):
        calls.append((k.get("inputs"), k.get("params")))
        return real(*a, **k)

    monkeypatch.setattr(batch, "wrench_vjp", spy)
    x2 = _dev(torch, planes).requires_grad_()
    loss_fn(batch.contact_wrench(x2, _dev(torch, prm)), _dev(torch, target)).backward()
    assert calls[-1] == (set(GROUP_NAMES), False)
    _check(x2.grad.cpu().numpy(), None, planes, prm, gbar, "state only", want=(xc.grad.numpy(), None))
    # per-plane leaves: only the twist planes require grad -> only the twist group
    leaves = [_dev(torch, planes[i]) for i in range(30)]
    for i in range(6):
        leaves[i].requires_grad_()
    loss_fn(batch.contact_wrench(leaves, _dev(torch, prm)), _dev(torch, target)).backward()
    assert calls[-1] == ({"twist"}, False)
    gx = np.zeros((30, n))
    gx[0:6] = torch.stack([leaves[i].grad for i in range(6)]).cpu().numpy()
    wx = np.zeros((30, n))
    wx[0:6] = xc.grad.numpy()[0:6]
    _check(gx, None, planes, prm, gbar, "twist leaves", want=(wx, None))
    assert all(leaves[i].grad is None for i in range(6, 30))


# --- C++ facade ---------------------------------------------------------------------------------------

def test_cpp_wrench_gradient():
    from bipedal_locomotion_framework_b200 import build
    build.build_cpp()
    r = subprocess.run([os.path.join(build.LIB_DIR, "ContactWrenchGradientUnitTests")],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "0 failure(s)" in r.stdout
