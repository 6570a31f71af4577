"""GPU parity tests for the end of FloatingBaseDynamicalSystem::dynamics
(src/System/src/FloatingBaseSystemDynamics.cpp:188-248 of the reference): the batched mass-matrix
solve (M + reg).llt().solve(known + torques) and the whole step from the bias forces on -- the CUDA
path through the C ABI against the CPU oracle on the same bits, the exact-rational golden fixture and
the reference's own source run over the KinDynComputations test double (oracle/_ref; its answers
through tests/reference_samples.py).
Tolerance: 1e-12 norm-wise relative per system (north_star) where the matrix's conditioning allows
it, c n eps cond(A) otherwise (parity.llt_tolerance)."""
import os

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from parity import TOL, assert_parity, llt_tolerance

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NTHREADS = max(1, (os.cpu_count() or 1))
PATH_LLT_WARP, PATH_LLT_BLOCK = 3, 4


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


@pytest.fixture(scope="module")
def dyn(batch):
    from bipedal_locomotion_framework_b200.system import FloatingBaseDynamicsBatch
    return FloatingBaseDynamicsBatch(batch)


@pytest.fixture(scope="module")
def so(oracle):
    from oracle import sys_oracle
    return sys_oracle


@pytest.fixture(scope="module")
def ref():
    import reference_samples   # what the reference build answers, pinned to stored samples
    return reference_samples


@pytest.fixture(scope="module")
def gd():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "dyn_exact_golden.npz")))


def _dev(torch, a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rel(got, ref):
    num = np.abs(np.asarray(got) - ref).max(axis=-1)
    den = np.maximum(np.abs(ref).max(axis=-1), 1e-300)
    return np.where(num == 0, 0.0, num / den)


def _last_path(batch):
    from bipedal_locomotion_framework_b200 import _capi
    return _capi.lib().blf_ccm_last_path(batch.handle.ptr)


def _case(nc, ns, seed, spread=0.0, with_tau=True, with_reg=False):
    rng = np.random.default_rng(seed)
    M = syn.make_mass_matrices(ns, nc, seed=seed + 1, spread=spread)
    known = rng.normal(size=(ns, nc)) * 30.0
    tau = rng.normal(size=(ns, nc - 6)) * 5.0 if (with_tau and nc > 6) else None
    reg = None
    if with_reg:
        reg = np.diag(10.0 ** rng.uniform(-4, -2, nc))
        reg[nc - 1, 0] = reg[0, nc - 1] = 1e-3
    return M, known, tau, reg


# --- the solve -------------------------------------------------------------------------------------

def test_mass_matrix_solve_matches_exact_rationals(torch, dyn, gd):
    """oracle/exact_golden_dyn.py: the solution is rational in the inputs, evaluated exactly."""
    for tag in gd["tags"]:
        M, known, acc, cond = (gd[f"{tag}_{k}"] for k in ("M", "known", "acc", "cond"))
        tau, reg = gd.get(f"{tag}_tau"), gd.get(f"{tag}_reg")
        x = dyn.solve(_dev(torch, M), _dev(torch, known), _dev(torch, tau), _dev(torch, reg)).cpu().numpy()
        err = rel(x, acc)
        assert (err <= llt_tolerance(known.shape[1], cond)).all(), (tag, err.max())
        easy = cond < 100
        if easy.any():
            assert err[easy].max() <= TOL, (tag, err[easy].max())


@pytest.mark.parametrize("nc", list(range(1, 50)) + [51, 52, 55, 59, 60, 63, 64, 65, 100, 128])
def test_mass_matrix_solve_vs_oracle_every_size(torch, batch, dyn, so, nc):
    """Every size class of the warp-level kernel (nc <= 64) and the block-level kernel above, a
    system count that fills no warp or CTA evenly; benign conditioning (cond < 4): flat 1e-12."""
    ns = 1003 if nc <= 49 else 131
    M, known, tau, reg = _case(nc, ns, 500 + nc, with_reg=bool(nc % 2))
    want = so.mass_matrix_solve(M, known, tau, reg, nthreads=NTHREADS)
    x = dyn.solve(_dev(torch, M), _dev(torch, known), _dev(torch, tau), _dev(torch, reg)).cpu().numpy()
    assert _last_path(batch) == (PATH_LLT_WARP if nc <= 64 else PATH_LLT_BLOCK)
    assert np.isfinite(x).all()
    err = rel(x, want)
    assert err.max() <= TOL, (int(np.argmax(err)), err.max())


@pytest.mark.parametrize("nc", [6, 12, 24, 29, 38, 59])
def test_mass_matrix_solve_tiny_batches(torch, dyn, so, nc):
    """1 .. 9 systems: partly filled groups of every lane layout (8, 4, 2, 1 systems per warp); the
    missing systems of a group are identity-padded inside the kernel and never written."""
    M, known, tau, reg = _case(nc, 9, 70 + nc, with_reg=True)
    want = so.mass_matrix_solve(M, known, tau, reg)
    dM, dk, dt, dr = (_dev(torch, a) for a in (M, known, tau, reg))
    for ns in range(1, 10):
        guard = torch.full((ns + 2, nc), 123.0, dtype=torch.float64, device="cuda")
        out = guard[1:ns + 1]
        dyn.solve(dM[:ns].contiguous(), dk[:ns].contiguous(), None if dt is None else dt[:ns].contiguous(), dr, out=out)
        assert rel(out.cpu().numpy(), want[:ns]).max() <= TOL, (nc, ns)
        assert bool((guard[0] == 123.0).all()) and bool((guard[ns + 1] == 123.0).all())   # nothing written outside


def test_warp_and_block_kernels_agree(torch, dyn, so):
    """The block-level kernel (forced on a second handle through BLF_CCM_TUNE_LLT_GENERAL, read when
    a handle is created) runs the same factorisation in the same order as the warp-level one; the
    back substitutions sum in different orders (butterfly over the lanes / sequential), so the two
    agree to rounding -- both within the tolerance against the oracle."""
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    from bipedal_locomotion_framework_b200.system import FloatingBaseDynamicsBatch
    os.environ["BLF_CCM_TUNE_LLT_GENERAL"] = "1"
    try:
        b2 = ContinuousContactModelBatch(0)
    finally:
        os.environ.pop("BLF_CCM_TUNE_LLT_GENERAL", None)
    gen = FloatingBaseDynamicsBatch(b2)
    for nc in (1, 3, 6, 7, 8, 12, 15, 16, 23, 29, 31, 38, 47, 59, 64):
        M, known, tau, reg = _case(nc, 301, 900 + nc, spread=1.0, with_reg=nc in (7, 29, 38))
        args = [_dev(torch, a) for a in (M, known, tau, reg)]
        fast = dyn.solve(*args).cpu().numpy()
        assert _last_path(dyn._b) == PATH_LLT_WARP
        slow = gen.solve(*args).cpu().numpy()
        assert _last_path(b2) == PATH_LLT_BLOCK
        want = so.mass_matrix_solve(M, known, tau, reg, nthreads=NTHREADS)
        tol = llt_tolerance(nc, np.linalg.cond(M if reg is None else M + reg, np.inf))
        assert (rel(fast, want) <= tol).all() and (rel(slow, want) <= tol).all(), nc
        assert (rel(fast, slow) <= tol).all(), nc


def test_mass_matrix_solve_in_place_and_stream(torch, dyn):
    """acc may alias known; the launch runs on the caller's current stream."""
    M, known, tau, _ = _case(29, 4097, 77)
    dM, dk, dt = (_dev(torch, a) for a in (M, known, tau))
    ref = dyn.solve(dM, dk, dt).clone()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        buf = dk.clone()
        out = dyn.solve(dM, buf, dt, out=buf)
    s.synchronize()
    assert out.data_ptr() == buf.data_ptr() and torch.equal(buf, ref)


def test_mass_matrix_solve_reads_only_the_lower_triangle(torch, dyn):
    M, known, tau, reg = _case(29, 513, 31, with_reg=True)
    x0 = dyn.solve(_dev(torch, M), _dev(torch, known), _dev(torch, tau), _dev(torch, reg))
    iu = np.triu_indices(29, 1)
    M2, reg2 = M.copy(), reg.copy()
    M2[:, iu[0], iu[1]] = np.nan
    reg2[iu] = np.nan
    x1 = dyn.solve(_dev(torch, M2), _dev(torch, known), _dev(torch, tau), _dev(torch, reg2))
    assert torch.equal(x0, x1)


@pytest.mark.parametrize("nc,spread", [(29, 1.5), (12, 2.0), (38, 1.0)])
def test_mass_matrix_solve_ill_conditioned(torch, dyn, so, nc, spread):
    """Inertias spread over 2-4 decades (cond up to ~1e8): forward error against the oracle within
    the bound both factorisations obey, and the backward error -- the residual -- at rounding level."""
    ns = 2001
    M, known, tau, _ = _case(nc, ns, 40 + nc, spread=spread)
    want = so.mass_matrix_solve(M, known, tau, nthreads=NTHREADS)
    x = dyn.solve(_dev(torch, M), _dev(torch, known), _dev(torch, tau)).cpu().numpy()
    cond = np.linalg.cond(M, np.inf)
    assert (rel(x, want) <= 2 * llt_tolerance(nc, cond)).all()
    rhs = known.copy()
    if tau is not None:
        rhs[:, 6:] += tau
    res = np.abs(np.einsum("sij,sj->si", M, x) - rhs).max(axis=1)
    scale = np.abs(M).sum(axis=2).max(axis=1) * np.abs(x).max(axis=1) + np.abs(rhs).max(axis=1)
    assert (res <= 8 * nc * 2.0 ** -52 * scale).all()


def test_not_positive_definite_gives_nan_for_that_system_only(torch, dyn, so):
    M, known, tau, _ = _case(12, 200, 9)
    M[17] = -M[17]
    M[101, 5, 5] = -1.0
    x = dyn.solve(_dev(torch, M), _dev(torch, known), _dev(torch, tau)).cpu().numpy()
    bad = np.isnan(x).any(axis=1)
    assert bad[17] and bad[101] and bad.sum() == 2
    want = so.mass_matrix_solve(M, known, tau)
    assert np.array_equal(np.isnan(want).any(axis=1), bad)      # the oracle: NaN for the same systems
    assert rel(x[~bad], want[~bad]).max() <= TOL


def test_mass_matrix_solve_rejects_bad_arguments(torch, batch, dyn):
    from bipedal_locomotion_framework_b200 import _capi
    L, h = _capi.lib(), batch.handle.ptr
    M, known, tau, _ = _case(8, 4, 1)
    dM, dk, dt = (_dev(torch, a) for a in (M, known, tau))
    out = torch.empty_like(dk)
    ok = lambda *a: L.blf_sys_mass_matrix_solve(h, *a)
    assert ok(4, 8, dM.data_ptr(), None, dk.data_ptr(), dt.data_ptr(), out.data_ptr(), None) == 0
    assert ok(0, 8, None, None, None, None, None, None) == 0                       # empty batch
    assert ok(-1, 8, dM.data_ptr(), None, dk.data_ptr(), None, out.data_ptr(), None) != 0
    assert ok(4, 0, dM.data_ptr(), None, dk.data_ptr(), None, out.data_ptr(), None) != 0
    assert ok(4, 129, dM.data_ptr(), None, dk.data_ptr(), None, out.data_ptr(), None) != 0
    assert ok(4, 8, None, None, dk.data_ptr(), None, out.data_ptr(), None) != 0
    assert ok(4, 8, dM.data_ptr() + 4, None, dk.data_ptr(), None, out.data_ptr(), None) != 0
    assert ok(4, 6, dM.data_ptr(), None, dk.data_ptr(), dt.data_ptr(), out.data_ptr(), None) != 0  # torques, no joints
    assert b"joint" in L.blf_ccm_last_error()


# --- the whole step: -bias + sum J^T wrench + torques, then the solve -------------------------------

def _acc_tolerance(M, x_ref, mag_rhs):
    """|dx| <= |M^-1| |d rhs| + LLT error: the right-hand side is a cancelling sum known only to
    1e-12 of the magnitude of its terms."""
    nc = M.shape[1]
    inv_norm = np.abs(np.linalg.inv(M)).sum(axis=2).max(axis=1)
    cond = inv_norm * np.abs(M).sum(axis=2).max(axis=1)
    return TOL * inv_norm * mag_rhs + llt_tolerance(nc, cond) * np.abs(x_ref).max(axis=1)


@pytest.mark.parametrize("cps,ncols,het,with_reg,spread", [
    (2, 29, False, False, 0.0), (2, 29, True, True, 1.0), (1, 6, False, False, 0.5),
    (4, 38, True, True, 0.5), (3, 12, False, True, 0.0)])
def test_floating_base_acceleration_vs_reference_build(torch, batch, dyn, ref, cps, ncols, het, with_reg, spread):
    """blf_sys_floating_base_acceleration against FloatingBaseDynamicalSystem::dynamics run from the
    reference's own FloatingBaseSystemDynamics.cpp over the KinDynComputations test double (mass
    matrices, bias forces, Jacobians and frame states injected; regularisation through
    setMassMatrixRegularization)."""
    ns = 2_001
    n = ns * cps
    st = syn.make_states(n, seed=85 + cps, heterogeneous=het)
    rng = np.random.default_rng(cps * 100 + ncols)
    J = rng.uniform(-1.0, 1.0, (n, 6, ncols))
    bias = rng.uniform(-50.0, 50.0, (ns, ncols))
    M, _, tau, reg = _case(ncols, ns, 60 + ncols, spread=spread, with_reg=with_reg)
    want, wref = ref.floating_base_dynamics(cps, st["twists"], st["poses"], st["null_poses"], J, bias, M,
                                            tau, reg, params=st["params"] if het else None,
                                            uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True,
                                            nthreads=NTHREADS)
    planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
    acc, wr = dyn.acceleration(cps, planes, _dev(torch, J), _dev(torch, bias), _dev(torch, M),
                               _dev(torch, tau), _dev(torch, reg),
                               param_planes=_dev(torch, st["params"].T) if het else None, want_wrench=True)
    assert_parity(wr.cpu().numpy().T, wref, "wrench")
    mag = np.abs(bias) + np.einsum("scrq,scr->sq", np.abs(J.reshape(ns, cps, 6, ncols)),
                                   np.abs(wref.reshape(ns, cps, 6)))
    if tau is not None:
        mag[:, 6:] += np.abs(tau)
    Meff = M if reg is None else M + reg
    tol = _acc_tolerance(Meff, want, mag.max(axis=1))
    err = np.abs(acc.cpu().numpy() - want).max(axis=1)
    assert (err <= tol).all(), (int(np.argmax(err / tol)), (err / tol).max())


def test_floating_base_acceleration_equals_its_two_steps(torch, batch, dyn):
    """One call = blf_ccm_generalized_force_soa on the negated bias + blf_sys_mass_matrix_solve,
    bit for bit; the bias array is left untouched."""
    from bipedal_locomotion_framework_b200.system import GeneralizedForceBatch
    cps, ncols, ns = 2, 29, 30_001
    st = syn.make_states(ns * cps, seed=3)
    rng = np.random.default_rng(8)
    J = _dev(torch, rng.uniform(-1, 1, (ns * cps, 6, ncols)))
    bias = _dev(torch, rng.uniform(-50, 50, (ns, ncols)))
    bias0 = bias.clone()
    M, _, tau, _ = _case(ncols, ns, 4)
    dM, dt = _dev(torch, M), _dev(torch, tau)
    planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
    acc = dyn.acceleration(cps, planes, J, bias, dM, dt)
    known = GeneralizedForceBatch(batch).run(cps, ncols, planes, J, -bias)
    assert torch.equal(acc, dyn.solve(dM, known, dt)) and torch.equal(bias, bias0)


def test_floating_base_acceleration_large_batch_residual(torch, batch, dyn):
    """409 600 systems (an MPC batch of 4096 samples x 100 steps), 2 contacts, 6 + 23 DoF: the
    size-independent property M acc = -bias + sum J^T wrench + torques, checked on the device."""
    cps, ncols, ns = 2, 29, 409_600
    planes = syn.make_planes_torch(ns * cps, batch.device, seed=12)[0]
    g = torch.Generator(device="cuda").manual_seed(5)
    J = torch.rand((ns * cps, 6, ncols), generator=g, device="cuda", dtype=torch.float64) * 2 - 1
    bias = (torch.rand((ns, ncols), generator=g, device="cuda", dtype=torch.float64) - 0.5) * 100
    tau = (torch.rand((ns, ncols - 6), generator=g, device="cuda", dtype=torch.float64) - 0.5) * 10
    A = torch.rand((ns, ncols, ncols), generator=g, device="cuda", dtype=torch.float64) * 2 - 1
    M = torch.bmm(A, A.transpose(1, 2)) / ncols
    del A
    M.diagonal(dim1=1, dim2=2).add_(0.5)
    M = torch.tril(M) + torch.tril(M, -1).transpose(1, 2)
    acc, wr = dyn.acceleration(cps, planes, J, bias, M, tau, want_wrench=True)
    assert bool(torch.isfinite(acc).all())
    W = wr.T.reshape(ns, cps, 6)
    rhs = -bias + torch.einsum("scrq,scr->sq", J.reshape(ns, cps, 6, ncols), W)
    rhs[:, 6:] += tau
    res = (torch.bmm(M, acc.unsqueeze(2)).squeeze(2) - rhs).abs().amax(dim=1)
    mag = bias.abs().amax(dim=1) + (J.reshape(ns, cps, 6, ncols).abs() * W.abs().unsqueeze(3)).sum(dim=(1, 2)).amax(dim=1)
    assert bool((res <= 1e-12 * (mag + M.abs().sum(dim=2).amax(dim=1) * acc.abs().amax(dim=1))).all())


# --- one ForwardEuler step of FloatingBaseDynamicalSystem ---------------------------------------------

def _rot(rng, scaled):
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return q * (1.0 + (0.02 * rng.normal() if scaled else 0.0))   # off the manifold: the Baumgarte term acts


@pytest.mark.parametrize("ncols,ns,rho", [(29, 5_003, 0.7), (29, 1_000, 0.0), (6, 4_099, 0.3), (12, 3_001, 2.0),
                                          (16, 777, 0.01), (38, 1_025, 0.5), (64, 131, 0.1), (128, 33, 0.0), (29, 4_096, 0.7), (7, 1, 0.2), (29, 2, 0.2), (23, 3, 0.0)])
@pytest.mark.parametrize("guard", [2, 1])
def test_floating_base_euler_step_vs_oracle(torch, dyn, so, ncols, ns, rho, guard):
    """blf_sys_floating_base_euler_step against the C oracle (itself bit-identical to the reference's
    ForwardEuler<FloatingBaseDynamicalSystem>): tiles of every size class, ragged and odd counts (last tile
    on the per-thread copy route), guard rows either side; two guard rows keep the arrays 16-byte aligned
    (bulk-copy route), one row leaves them 8-byte aligned (per-thread route)."""
    rng = np.random.default_rng(ncols + ns)
    dT = 0.01
    acc = rng.normal(size=(ns, ncols)) * 30.0
    nu = rng.normal(size=(ns, ncols))
    jp = rng.normal(size=(ns, ncols - 6)) if ncols > 6 else None
    p = rng.normal(size=(ns, 3))
    R = np.stack([_rot(rng, i % 2 == 0) for i in range(ns)])
    wv, wq, wp, wR = so.floating_base_euler_step(rho, dT, acc, nu, jp, p, R, nthreads=NTHREADS)
    pad = lambda x: None if x is None else torch.from_numpy(np.concatenate([np.full((guard,) + x.shape[1:], 7.5), x,
                                                                           np.full((guard,) + x.shape[1:], 7.5)])).cuda()
    dv, dq, dp_, dR = pad(nu), pad(jp), pad(p), pad(R.reshape(ns, 9))
    view = lambda x: None if x is None else x[guard:ns + guard]
    dyn.euler_step(rho, dT, _dev(torch, acc), view(dv), view(dq), view(dp_), view(dR))
    for got, want in ((dv, wv), (dq, wq), (dp_, wp), (dR, wR.reshape(ns, 9))):
        if got is None:
            continue
        g = got.cpu().numpy()
        assert (g[:guard] == 7.5).all() and (g[-guard:] == 7.5).all()        # nothing written outside
        assert rel(g[guard:-guard], want).max() <= TOL
    assert rel(dR.cpu().numpy()[guard:-guard].reshape(ns, 3, 3), wR).max() <= TOL    # row by row


def test_floating_base_whole_step_vs_reference_build(torch, batch, dyn, ref):
    """Acceleration + Euler step through the C ABI against ForwardEuler<FloatingBaseDynamicalSystem>
    run from the reference's own sources over the test double."""
    cps, ncols, ns, rho, dT = 2, 29, 1_501, 0.7, 0.01
    st = syn.make_states(ns * cps, seed=17)
    rng = np.random.default_rng(99)
    J = rng.uniform(-1.0, 1.0, (ns * cps, 6, ncols))
    bias = rng.uniform(-50.0, 50.0, (ns, ncols))
    M, _, tau, _ = _case(ncols, ns, 21)
    nu = rng.normal(size=(ns, ncols))
    jp = rng.normal(size=(ns, ncols - 6))
    p = rng.normal(size=(ns, 3))
    R = np.stack([_rot(rng, True) for _ in range(ns)])
    racc, rv, rq, rp, rR = ref.floating_base_euler_step(cps, st["twists"], st["poses"], st["null_poses"], J, bias, M,
                                                        rho, dT, nu, jp, p, R, joint_torques=tau,
                                                        uniform=syn.REFERENCE_TEST_PARAMS, nthreads=NTHREADS)
    planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
    acc = dyn.acceleration(cps, planes, _dev(torch, J), _dev(torch, bias), _dev(torch, M), _dev(torch, tau))
    dv, dq, dp_, dR = (_dev(torch, x) for x in (nu, jp, p, R.reshape(ns, 9)))
    dyn.euler_step(rho, dT, acc, dv, dq, dp_, dR)
    # the velocity inherits the acceleration's tolerance scaled by dT; the rest is elementwise
    mag = np.abs(bias).max(axis=1) + np.abs(J.reshape(ns, cps, 6, ncols)).sum(axis=(1, 2)).max(axis=1) * 1e3
    tol_acc = _acc_tolerance(M, racc, mag)
    assert (np.abs(acc.cpu().numpy() - racc).max(axis=1) <= tol_acc).all()
    assert (np.abs(dv.cpu().numpy() - rv).max(axis=1) <= tol_acc * dT + TOL * np.abs(rv).max(axis=1)).all()
    assert rel(dq.cpu().numpy(), rq).max() <= TOL and rel(dp_.cpu().numpy(), rp).max() <= TOL
    assert rel(dR.cpu().numpy().reshape(ns, 3, 3), rR).max() <= TOL


def test_floating_base_euler_step_rejects_bad_arguments(torch, batch):
    from bipedal_locomotion_framework_b200 import _capi
    L, h = _capi.lib(), batch.handle.ptr
    z = lambda *s: torch.zeros(s, dtype=torch.float64, device="cuda")
    acc, nu, jp, p, R = z(4, 8), z(4, 8), z(4, 2), z(4, 3), z(4, 9)
    R[:, 0] = R[:, 4] = R[:, 8] = 1.0
    f = lambda *a: L.blf_sys_floating_base_euler_step(h, *a)
    assert f(4, 8, 0.1, 0.01, acc.data_ptr(), nu.data_ptr(), jp.data_ptr(), p.data_ptr(), R.data_ptr(), None) == 0
    assert f(0, 8, 0.1, 0.01, None, None, None, None, None, None) == 0
    assert f(4, 5, 0.1, 0.01, acc.data_ptr(), nu.data_ptr(), jp.data_ptr(), p.data_ptr(), R.data_ptr(), None) != 0
    assert f(4, 8, 0.1, 0.01, acc.data_ptr(), nu.data_ptr(), None, p.data_ptr(), R.data_ptr(), None) != 0
    assert f(4, 8, 0.1, 0.01, nu.data_ptr(), nu.data_ptr(), jp.data_ptr(), p.data_ptr(), R.data_ptr(), None) != 0
    assert f(4, 6, 0.1, 0.01, acc.data_ptr(), nu.data_ptr(), None, p.data_ptr(), R.data_ptr(), None) == 0


def test_floating_base_euler_step_large_batch_properties(torch, batch, dyn):
    """2^21 systems x 29 unknowns (2.6 GB of state, well past L2), checked on the device: the velocity, joint
    and position updates against the same multiply-add in torch (two roundings there, one here: an ulp of the larger term), the
    rotations bit for bit against the kinematics' own batched Euler step (blf_sys_kinematics_euler_step_soa,
    another kernel around the same device function), and the step is a pure function of its inputs."""
    from bipedal_locomotion_framework_b200.system import KinematicsBatch
    ns, nc, rho, dT = 1 << 21, 29, 0.7, 0.01
    g = torch.Generator(device="cuda").manual_seed(5)
    rnd = lambda *s: torch.rand(s, dtype=torch.float64, device="cuda", generator=g) * 2 - 1
    acc, nu, jp, p = rnd(ns, nc) * 30, rnd(ns, nc), rnd(ns, nc - 6), rnd(ns, 3)
    qt = rnd(ns, 4)
    w, x, y, z = (qt / qt.norm(dim=1, keepdim=True)).unbind(1)          # unit quaternions -> rotations
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], dim=1)
    R = (R * (1.0 + 0.02 * rnd(ns, 1))).contiguous()                     # off the manifold: the Baumgarte term acts
    v1, j1, p1, R1 = nu.clone(), jp.clone(), p.clone(), R.clone()
    dyn.euler_step(rho, dT, acc, v1, j1, p1, R1)
    # x + d * dT: one rounding here (fma), two in torch -- they differ by at most an ulp of the larger term
    close = lambda got, x, d: bool(((got - (x + d * dT)).abs() <= 2.3e-16 * (x.abs() + (d * dT).abs())).all())
    assert close(v1, nu, acc) and close(j1, jp, nu[:, 6:]) and close(p1, p, nu[:, :3])
    kb = KinematicsBatch(0, batch.handle)
    tw = nu[:, :6].t().contiguous()
    kp, kR = p.t().contiguous(), R.t().contiguous()
    kb.prepare_euler_step(rho, dT, tw, kp, kR)()
    assert torch.equal(kp.t(), p1) and bool(((kR.t() - R1).abs() <= 1e-14).all())
    v2, j2, p2, R2 = nu.clone(), jp.clone(), p.clone(), R.clone()
    dyn.euler_step(rho, dT, acc, v2, j2, p2, R2)
    assert torch.equal(v1, v2) and torch.equal(j1, j2) and torch.equal(p1, p2) and torch.equal(R1, R2)


@pytest.mark.parametrize("cps,ncols,het,with_reg", [(2, 29, False, False), (2, 29, True, True), (1, 6, False, False),
                                                    (3, 12, True, False)])
def test_facade_class_vs_reference_class(torch, ref, cps, ncols, het, with_reg):
    """The PRODUCT's C++ class System::FloatingBaseDynamicalSystem + ForwardEuler (GPU; through
    oracle/refbuild/facade_glue/facade_fbd_driver.cpp) against the REFERENCE'S own class compiled from its
    sources (CPU; ref_driver.cpp), both driven through their public methods on the same arrays:
    dynamics() and one integrate(0, dT) per system."""
    ns, rho, dT = 40, 0.7, 0.01
    st = syn.make_states(ns * cps, seed=60 + ncols, heterogeneous=het)
    rng = np.random.default_rng(61 + ncols)
    J = rng.uniform(-1.0, 1.0, (ns * cps, 6, ncols))
    bias = rng.uniform(-50.0, 50.0, (ns, ncols))
    M = syn.make_mass_matrices(ns, ncols, seed=5 + ncols, spread=0.5)
    tau = rng.uniform(-5.0, 5.0, (ns, ncols - 6)) if ncols > 6 else None
    reg = np.diag(rng.uniform(0.01, 0.2, ncols)) if with_reg else None
    nu = rng.normal(size=(ns, ncols))
    jp = rng.normal(size=(ns, ncols - 6)) if ncols > 6 else None
    p = rng.normal(size=(ns, 3))
    R = np.stack([_rot(rng, True) for _ in range(ns)])
    kw = dict(joint_torques=tau, reg=reg, params=st["params"] if het else None, uniform=syn.REFERENCE_TEST_PARAMS)
    args = (cps, st["twists"], st["poses"], st["null_poses"], J, bias, M, rho, dT, nu, jp, p, R)
    racc, rv, rq, rp, rR = ref.floating_base_euler_step(*args, nthreads=NTHREADS, **kw)
    facc, fv, fq, fp, fR = ref.facade_floating_base_euler_step(*args, **kw)
    mag = np.abs(bias).max(axis=1) + np.abs(J.reshape(ns, cps, 6, ncols)).sum(axis=(1, 2)).max(axis=1) * 1e3
    tol_acc = _acc_tolerance(M if reg is None else M + reg, racc, mag)
    assert (np.abs(facc - racc).max(axis=1) <= tol_acc).all()
    assert (np.abs(fv - rv).max(axis=1) <= tol_acc * dT + TOL * np.abs(rv).max(axis=1)).all()
    assert rel(fp, rp).max() <= TOL and rel(fR, rR).max() <= TOL
    if ncols > 6:
        assert rel(fq, rq).max() <= TOL


def _place(torch, a, shift):
    """`a` on the device, `shift` doubles into a fresh buffer: 16-byte aligned (0) or 8 bytes off (1)."""
    if a is None:
        return None
    buf = torch.empty(a.size + 2, dtype=torch.float64, device="cuda")
    v = buf[shift:shift + a.size].view(a.shape)
    v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    assert v.data_ptr() % 16 == 8 * shift
    return v


@pytest.mark.parametrize("nc,ns,with_reg", [(6, 4_099, False), (8, 2_051, True), (12, 4_099, False), (12, 1_003, True),
                                            (12, 5, False), (6, 1, False), (10, 3_001, True), (14, 2_003, False)])
def test_mass_matrix_solve_bulk_and_per_thread_fill_agree(torch, dyn, so, nc, ns, with_reg):
    """6, 8, 10, 12 and 14 unknowns on 16-byte aligned arrays take the bulk-copy fill (dense tiles, three bulk copies per
    system); the same arrays 8 bytes off take the per-thread copies (packed tiles).  Same arithmetic on the same
    operands: bit-identical results, both within 1e-12 of the oracle; ragged last groups; in place."""
    M, known, tau, reg = _case(nc, ns, 900 + nc + ns, with_reg=with_reg)
    want = so.mass_matrix_solve(M, known, tau, reg, nthreads=NTHREADS)

    def run(shift):
        dM, dk, dt = (_place(torch, a, shift) for a in (M, known, tau))
        x = dyn.solve(dM, dk, dt, _dev(torch, reg)).cpu().numpy()
        dyn.solve(dM, dk, dt, _dev(torch, reg), out=dk)          # in place: acc may alias known
        assert np.array_equal(dk.cpu().numpy(), x)
        return x

    bulk, per_thread = run(0), run(1)
    assert np.array_equal(bulk, per_thread)
    assert rel(bulk, want).max() <= TOL


# --- batches the solve's persistent warps take in several passes -----------------------------------------

def _multi_pass(torch, nc):
    """(ns, W, SPW) for a batch that every warp of the warp-level solve takes in three passes or more.
    A warp solves SPW systems at a time (8 up to 15 unknowns, 4 up to 31, 2 up to 47, 1 up to 64: the lane
    classes of csrc/dyn_kernels.cu) and strides over the groups of SPW by the number of warps launched.
    The launcher caps the grid at the CTAs of 64 threads that are resident at once, so no launch has more
    than W = SMs x max threads per SM / 32 warps, whatever the occupancy, and 3 W SPW systems need three
    passes.  The extra 37 SPW + (SPW + 1) // 2 systems make the last group ragged (SPW > 1) and the group
    count 3 W + 38, no multiple of W.  148-SM B200: 227 k systems up to 15 unknowns, 114 k up to 31,
    57 k up to 47, 28 k up to 64."""
    p = torch.cuda.get_device_properties(0)
    spw = 8 if nc <= 15 else 4 if nc <= 31 else 2 if nc <= 47 else 1
    w = p.multi_processor_count * p.max_threads_per_multi_processor // 32
    return 3 * w * spw + 37 * spw + (spw + 1) // 2, w, spw


BULK_ORDERS = (6, 8, 10, 12, 14)   # even orders that fill a 4-lane class exactly: the bulk-copy fill when aligned
MULTI_PASS_ORDERS = BULK_ORDERS + (5, 9, 15) + (16, 23, 24, 29, 31) + (32, 38, 47) + (48, 59, 64)


@pytest.mark.parametrize("nc,with_reg", [(nc, i % 2 == 1) for i, nc in enumerate(MULTI_PASS_ORDERS)])
def test_mass_matrix_solve_multi_pass_vs_oracle(torch, batch, dyn, so, nc, with_reg):
    """Every lane class (4, 8, 16, 32 lanes per system; 24 unknowns: the right-hand side as a column) on a
    batch its warps take in three passes or more, so the tiles are refilled for the next group while the
    current one is factorised: within 1e-12 of the oracle, nothing written outside the output, in place =
    out of place bit for bit.  The even orders up to 14 run twice, 16-byte aligned (bulk-copy refills on the
    warp's mbarrier) and 8 bytes off (per-thread copies): bit-identical."""
    ns = _multi_pass(torch, nc)[0]
    M, known, tau, reg = _case(nc, ns, 1300 + nc, with_reg=with_reg)
    want = so.mass_matrix_solve(M, known, tau, reg, nthreads=NTHREADS)
    dr = _dev(torch, reg)

    def run(shift):
        dM, dk, dt = (_place(torch, a, shift) for a in (M, known, tau))
        guard = torch.full((ns + 2, nc), 123.0, dtype=torch.float64, device="cuda")
        x = dyn.solve(dM, dk, dt, dr, out=guard[1:ns + 1])
        assert _last_path(batch) == PATH_LLT_WARP
        assert bool((guard[0] == 123.0).all()) and bool((guard[ns + 1] == 123.0).all())   # nothing written outside
        dyn.solve(dM, dk, dt, dr, out=dk)          # in place, as the whole step solves
        assert torch.equal(dk, x)
        return x.cpu().numpy()

    x = run(0)
    assert np.isfinite(x).all()
    err = rel(x, want)
    assert err.max() <= TOL, (ns, int(np.argmax(err)), err.max())
    if nc in BULK_ORDERS:
        y = run(1)
        assert np.array_equal(y, x), (ns, int(np.argmax(np.abs(y - x).max(axis=1))))


@pytest.mark.parametrize("nc", [12, 14, 15, 29, 38])
def test_mass_matrix_solve_position_invariant_across_passes(torch, dyn, nc):
    """A system's arithmetic does not depend on where it sits in the batch: the systems of a multi-pass batch
    equal, bit for bit, the same systems solved as a batch of their own that takes one pass -- the first
    ones, the ones from W SPW on (no earlier than the second pass) and the ragged tail.  Catches a refill of
    the wrong group or a stale tile even where its error would fit inside 1e-12.  Slices of even orders
    stay 16-byte aligned: 12 and 14 take the bulk-copy fill in both calls."""
    ns, w, spw = _multi_pass(torch, nc)
    M, known, tau, reg = _case(nc, ns, 1400 + nc, with_reg=True)
    dM, dk, dt, dr = (_dev(torch, a) for a in (M, known, tau, reg))
    x = dyn.solve(dM, dk, dt, dr)
    # 2 x SMs groups: a warp per group, one pass, since at least one CTA of two warps per SM is resident
    c = 2 * torch.cuda.get_device_properties(0).multi_processor_count * spw - 1
    for a in (0, w * spw, ns - c):
        part = dyn.solve(dM[a:a + c], dk[a:a + c], None if dt is None else dt[a:a + c], dr)
        assert torch.equal(part, x[a:a + c]), (ns, a)


@pytest.mark.parametrize("nc", [12, 38])
def test_not_positive_definite_stays_local_across_passes(torch, dyn, nc):
    """Systems that are not positive definite in the first pass, in a later one and in the ragged last group
    give NaN; every other system is bit-identical to the batch without them.  38 unknowns (16-lane groups,
    blocked back substitution) read entries of the diagonal-block buffer that only earlier passes wrote --
    NaN after a bad system -- into lanes that hold no unknown: harmless, and pinned here."""
    ns, w, spw = _multi_pass(torch, nc)
    M, known, tau, reg = _case(nc, ns, 1500 + nc, with_reg=True)
    dk, dt, dr = (_dev(torch, a) for a in (known, tau, reg))
    x0 = dyn.solve(_dev(torch, M), dk, dt, dr).cpu().numpy()
    bad = [3, 2 * w * spw + 5, ns - 1]
    M[bad[0]] = -M[bad[0]]
    M[bad[1], 5, 5] = -1.0
    M[bad[2], nc - 1, nc - 1] = -1.0
    x1 = dyn.solve(_dev(torch, M), dk, dt, dr).cpu().numpy()
    assert np.array_equal(np.flatnonzero(np.isnan(x1).any(axis=1)), bad), ns
    ok = np.ones(ns, dtype=bool)
    ok[bad] = False
    assert np.array_equal(x1[ok], x0[ok]), ns


@pytest.mark.parametrize("ncols,het,with_reg", [(12, False, True), (6, True, False)])
def test_floating_base_acceleration_multi_pass_vs_oracle(torch, batch, dyn, so, ncols, het, with_reg):
    """blf_sys_floating_base_acceleration at the small sizes of the benchmark, 2 contacts, on a batch whose
    solve takes three passes or more: the solve runs in place on the bulk-copy fill.  Against the C oracle
    within the conditioning-aware bound of the whole step."""
    cps = 2
    ns = _multi_pass(torch, ncols)[0]
    n = ns * cps
    st = syn.make_states(n, seed=160 + ncols, heterogeneous=het)
    rng = np.random.default_rng(161 + ncols)
    J = rng.uniform(-1.0, 1.0, (n, 6, ncols))
    bias = rng.uniform(-50.0, 50.0, (ns, ncols))
    M, _, tau, reg = _case(ncols, ns, 162 + ncols, with_reg=with_reg)
    planes = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])
    prm = st["params"].T if het else None
    want, wr = so.floating_base_acceleration(cps, planes, J, bias, M, tau, reg, param_planes=prm,
                                             uniform=syn.REFERENCE_TEST_PARAMS, want_wrench=True, nthreads=NTHREADS)
    acc = dyn.acceleration(cps, _dev(torch, planes), _dev(torch, J), _dev(torch, bias), _dev(torch, M),
                           _dev(torch, tau), _dev(torch, reg), param_planes=_dev(torch, prm))
    assert _last_path(batch) == PATH_LLT_WARP
    mag = np.abs(bias) + np.einsum("scrq,scr->sq", np.abs(J.reshape(ns, cps, 6, ncols)),
                                   np.abs(wr.T.reshape(ns, cps, 6)))
    if tau is not None:
        mag[:, 6:] += np.abs(tau)
    tol = _acc_tolerance(M if reg is None else M + reg, want, mag.max(axis=1))
    err = np.abs(acc.cpu().numpy() - want).max(axis=1)
    assert (err <= tol).all(), (ns, int(np.argmax(err / tol)), (err / tol).max())
