"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same
bits, against the exact-rational golden fixtures, and through size-independent properties at
BASELINE.json's full sizes.  Tolerance: 1e-12 norm-wise relative per 3-vector block (north_star),
structural zeros of the control matrix exactly +0.0."""
import os

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import synthetic as syn
from parity import TOL, assert_ctrl_structure, assert_parity

pytestmark = pytest.mark.gpu

NTHREADS = max(1, (os.cpu_count() or 1))
W, A, Cc, R = 1, 2, 4, 8
FULL = W | A | Cc
KEYS = {W: "wrench", A: "autodyn", Cc: "ctrl", R: "regressor"}


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


def _soa_inputs(torch, st):
    planes = _dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]))
    prm = _dev(torch, st["params"].T) if st["params"] is not None else None
    return planes, prm


def _soa_out_to_aos(out):
    r = {}
    for key in ("wrench", "autodyn", "regressor"):
        r[key] = None if out[key] is None else out[key].cpu().numpy().T.copy()
    r["ctrl"] = None if out["ctrl"] is None else out["ctrl"].cpu().numpy()
    return r


def _aos_out(out):
    return {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}


def _check(got, ref, mask, what):
    worst = 0.0
    for bit, key in KEYS.items():
        if mask & bit:
            e, _ = assert_parity(got[key], ref[key], key, what=what + " ")
            worst = max(worst, e)
    if mask & Cc:
        assert_ctrl_structure(got["ctrl"])
    return worst


# --- golden fixtures -------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", ["soa", "aos", "host"])
def test_golden_vectors(torch, batch, golden, layout):
    g = golden
    st = {"twists": g["twists"], "poses": g["poses"], "null_poses": g["null_poses"],
          "params": g["params"]}
    mask = FULL | R
    if layout == "soa":
        planes, prm = _soa_inputs(torch, st)
        got = _soa_out_to_aos(batch.evaluate_soa(planes, prm, mask))
    elif layout == "aos":
        got = _aos_out(batch.evaluate_aos(_dev(torch, st["twists"]), _dev(torch, st["poses"]),
                                          _dev(torch, st["null_poses"]), _dev(torch, st["params"]),
                                          mask))
    else:
        got = batch.evaluate_host(st["twists"], st["poses"], st["null_poses"], st["params"], mask)
    for key in ("wrench", "autodyn", "ctrl"):
        assert_parity(got[key], g[key], key, what=f"golden/{layout} ")
    floor = np.full(g["twists"].shape[0], 1e-300)
    floor[8] = 1e-6  # pose == null pose: the block cancels to exactly 0 (see test_oracle.py)
    assert_parity(got["regressor"], g["regressor"], "regressor", floor=floor)
    assert_ctrl_structure(got["ctrl"])


# --- BASELINE.json configs ---------------------------------------------------------------------------

def test_config2_one_million_wrench_only_soa(torch, batch, oracle):
    """configs[1]: 2^20 random states, wrench only, uniform parameters, SoA."""
    st = syn.make_states(1 << 20, seed=42 + 2)
    planes, _ = _soa_inputs(torch, st)
    got = _soa_out_to_aos(batch.evaluate_soa(planes, None, W))
    assert batch.handle.last_path == 1  # BLF_CCM_PATH_BULK
    ref = oracle.eval_batch_states(st, mask=W, nthreads=NTHREADS)
    _check(got, ref, W, "config2")


@pytest.mark.parametrize("layout", ["soa", "aos"])
def test_config3_mpc_rollout_batch_full(torch, batch, oracle, layout):
    """configs[2]: 2 feet x 4096 samples x 100 steps, wrench + autonomous dynamics + control."""
    n = 2 * 4096 * 100
    st = syn.make_states(n, seed=42 + 3)
    ref = oracle.eval_batch_states(st, mask=FULL, nthreads=NTHREADS)
    if layout == "soa":
        planes, _ = _soa_inputs(torch, st)
        got = _soa_out_to_aos(batch.evaluate_soa(planes, None, FULL))
    else:
        got = _aos_out(batch.evaluate_aos(_dev(torch, st["twists"]), _dev(torch, st["poses"]),
                                          _dev(torch, st["null_poses"]), None, FULL))
    assert batch.handle.last_path == 1
    _check(got, ref, FULL, f"config3/{layout}")


@pytest.mark.parametrize("layout", ["soa", "aos"])
def test_config4_heterogeneous_parameters(torch, batch, oracle, layout):
    """configs[3] at a size the oracle finishes in seconds: per-contact length/width/spring/damper."""
    n = (1 << 18) + 37
    st = syn.make_states(n, seed=42 + 4, heterogeneous=True)
    ref = oracle.eval_batch_states(st, mask=FULL | R, nthreads=NTHREADS)
    if layout == "soa":
        planes, prm = _soa_inputs(torch, st)
        got = _soa_out_to_aos(batch.evaluate_soa(planes, prm, FULL | R))
    else:
        got = _aos_out(batch.evaluate_aos(_dev(torch, st["twists"]), _dev(torch, st["poses"]),
                                          _dev(torch, st["null_poses"]), _dev(torch, st["params"]),
                                          FULL | R))
    _check(got, ref, FULL | R, f"config4/{layout}")


def test_host_pipeline_matches_device_path(torch, batch, oracle):
    """blf_ccm_eval_batch_host (chunked, overlapped copies) over several chunks + a ragged tail."""
    n = 3 * 32768 + 4321
    st = syn.make_states(n, seed=11, heterogeneous=True)
    ref = oracle.eval_batch_states(st, mask=FULL, nthreads=NTHREADS)
    got = batch.evaluate_host(st["twists"], st["poses"], st["null_poses"], st["params"], FULL)
    _check(got, ref, FULL, "host")
    got_u = batch.evaluate_host(st["twists"], st["poses"], st["null_poses"], None, W)
    ref_u = oracle.eval_batch_aos(st["twists"], st["poses"], st["null_poses"], None,
                                  syn.REFERENCE_TEST_PARAMS, W, NTHREADS)
    _check(got_u, ref_u, W, "host/uniform")


# --- edge cases ---------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [0, 1, 2, 31, 32, 33, 63, 64, 65, 127, 129, 1000])
@pytest.mark.parametrize("layout", ["soa", "aos"])
def test_ragged_sizes(torch, batch, oracle, n, layout):
    st = syn.make_states(max(n, 1), seed=5)
    st = {k: (v[:n] if isinstance(v, np.ndarray) else v) for k, v in st.items()}
    if layout == "soa":
        planes = torch.empty((30, n), dtype=torch.float64, device="cuda")
        if n:
            planes.copy_(_dev(torch, syn.aos_to_planes(st["twists"], st["poses"],
                                                       st["null_poses"])))
        got = _soa_out_to_aos(batch.evaluate_soa(planes, None, FULL | R))
    else:
        mk = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        got = _aos_out(batch.evaluate_aos(mk(st["twists"]), mk(st["poses"]), mk(st["null_poses"]),
                                          None, FULL | R))
    if n == 0:
        return
    ref = oracle.eval_batch_aos(st["twists"], st["poses"], st["null_poses"], None,
                                syn.REFERENCE_TEST_PARAMS, FULL | R, 1)
    _check(got, ref, FULL | R, f"n={n}/{layout}")


@pytest.mark.parametrize("mask", list(range(1, 16)))
def test_every_output_mask_and_untouched_outputs(torch, batch, oracle, mask):
    """Each of the 15 getter combinations; outputs not requested are not written."""
    n = 777
    st = syn.make_states(n, seed=9)
    ref = oracle.eval_batch_states(st, mask=mask, nthreads=1)
    planes, _ = _soa_inputs(torch, st)
    sentinel = -123.25
    out = batch.alloc_soa_outputs(n, 15)
    for v in out.values():
        v.fill_(sentinel)
    call_out = {key: (out[key] if mask & bit else None) for bit, key in KEYS.items()}
    batch.evaluate_soa(planes, None, mask, out=call_out)
    got = _soa_out_to_aos(out)
    _check(got, ref, mask, f"mask={mask}")
    for bit, key in KEYS.items():
        if not mask & bit:
            assert np.all(got[key] == sentinel)
    # AoS flavour of the same mask
    aout = batch.evaluate_aos(_dev(torch, st["twists"]), _dev(torch, st["poses"]),
                              _dev(torch, st["null_poses"]), None, mask)
    _check(_aos_out(aout), ref, mask, f"mask={mask}/aos")


def test_dead_planes_may_be_null(torch, batch, oracle):
    """Planes that cannot affect the requested outputs are never read (NULL is accepted)."""
    import ctypes as C
    from bipedal_locomotion_framework_b200 import _capi
    n = 4096
    st = syn.make_states(n, seed=13)
    planes, _ = _soa_inputs(torch, st)
    ptrs = [planes[i].data_ptr() for i in range(30)]
    for dead in (11, 14, 23, 26, 29):   # R02, R12 (autodyn only) and R0's third column
        ptrs[dead] = None
    arr = (C.c_void_p * 30)(*ptrs)
    w = torch.empty((6, n), dtype=torch.float64, device="cuda")
    c = torch.empty((n, 36), dtype=torch.float64, device="cuda")
    wp = (C.c_void_p * 6)(*[w[i].data_ptr() for i in range(6)])
    rc = _capi.lib().blf_ccm_eval_batch_soa(batch.handle.ptr, n, arr, None, W | Cc, wp, None,
                                            c.data_ptr(), None, None)
    assert rc == 0, _capi.lib().blf_ccm_last_error()
    torch.cuda.synchronize()
    ref = oracle.eval_batch_states(st, mask=W | Cc)
    assert_parity(w.cpu().numpy().T, ref["wrench"], "wrench")
    assert_parity(c.cpu().numpy(), ref["ctrl"], "ctrl")
    # ...but a live plane that is NULL is an argument error, not a crash
    ptrs[17] = None
    arr = (C.c_void_p * 30)(*ptrs)
    rc = _capi.lib().blf_ccm_eval_batch_soa(batch.handle.ptr, n, arr, None, W, wp, None, None,
                                            None, None)
    assert rc == _capi.ERR_INVALID_ARG


@pytest.mark.parametrize("layout", ["soa", "aos"])
def test_eight_byte_aligned_buffers_take_the_checked_64bit_path(torch, batch, oracle, layout):
    n = 5000
    st = syn.make_states(n, seed=21, heterogeneous=True)
    ref = oracle.eval_batch_states(st, mask=FULL, nthreads=1)
    if layout == "soa":
        # shift every plane by one double: rows start 8-byte but not 16-byte aligned
        big = torch.empty((30, n + 2), dtype=torch.float64, device="cuda")
        planes = big[:, 1:n + 1]
        planes.copy_(_dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])))
        assert planes[0].data_ptr() % 16 == 8
        prm = _dev(torch, st["params"].T)
        out = batch.alloc_soa_outputs(n, FULL)
        cbuf = torch.empty(n * 36 + 1, dtype=torch.float64, device="cuda")
        out["ctrl"] = cbuf[1:].view(n, 36)          # dense 6x6 array 8- but not 16-byte aligned
        assert out["ctrl"].data_ptr() % 16 == 8
        got = _soa_out_to_aos(batch.evaluate_soa(planes, prm, FULL, out=out))
    else:
        def shifted(a):
            buf = torch.empty(a.size + 1, dtype=torch.float64, device="cuda")
            v = buf[1:].view(a.shape)
            v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
            assert v.data_ptr() % 16 == 8
            return v
        got = _aos_out(batch.evaluate_aos(shifted(st["twists"]), shifted(st["poses"]),
                                          shifted(st["null_poses"]), _dev(torch, st["params"]),
                                          FULL))
    assert batch.handle.last_path == 2  # BLF_CCM_PATH_DIRECT64: dispatched, reported, same results
    _check(got, ref, FULL, f"unaligned/{layout}")


def test_uninitialised_handle_is_an_error(torch):
    from bipedal_locomotion_framework_b200 import _capi
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    b = ContinuousContactModelBatch(0)
    planes = torch.zeros((30, 64), dtype=torch.float64, device="cuda")
    with pytest.raises(_capi.BlfCcmError) as e:
        b.evaluate_soa(planes, None, W)
    assert e.value.code == _capi.ERR_NOT_INITIALIZED


# --- properties at full size ------------------------------------------------------------------------

def test_full_size_properties(torch, batch):
    """At configs[2] size without the oracle: (i) AoS and SoA entry points agree, (ii) the wrench
    is the regressor times [k; b] (ContinousContactModelTest.cpp:107-124), (iii) control-matrix
    structure, (iv) determinism (two runs bit-identical)."""
    n = 2 * 4096 * 100
    st = syn.make_states(n, seed=77)
    planes, _ = _soa_inputs(torch, st)
    a = batch.evaluate_soa(planes, None, FULL | R)
    b2 = batch.evaluate_soa(planes, None, FULL | R)
    for k in a:
        assert torch.equal(a[k], b2[k])
    aos = batch.evaluate_aos(_dev(torch, st["twists"]), _dev(torch, st["poses"]),
                             _dev(torch, st["null_poses"]), None, FULL | R)
    soa_as_aos = _soa_out_to_aos(a)
    aos_np = _aos_out(aos)
    for bit, key in KEYS.items():
        assert_parity(aos_np[key], soa_as_aos[key], key, tol=1e-13, what="aos vs soa ")
    _, _, k, bb = syn.REFERENCE_TEST_PARAMS
    Y = soa_as_aos["regressor"].reshape(n, 6, 2)
    via_regressor = Y @ np.array([k, bb])
    assert_parity(via_regressor, soa_as_aos["wrench"], "wrench", tol=1e-11)
    assert_ctrl_structure(soa_as_aos["ctrl"])
    g = soa_as_aos["ctrl"].reshape(n, 6, 6)
    assert np.array_equal(g[:, 3:, 3:], g[:, 3:, 3:].transpose(0, 2, 1))  # symmetric block


# --- per-instance facade: the reference's own test against the GPU ---------------------------------

def _handler(k=2000.0, b=100.0, L=0.12, Wd=0.09):
    from bipedal_locomotion_framework_b200.contact_models import StdImplementation
    h = StdImplementation()
    h.setParameter("spring_coeff", k)
    h.setParameter("damper_coeff", b)
    h.setParameter("length", L)
    h.setParameter("width", Wd)
    return h


def _rodrigues(w):
    th = np.linalg.norm(w)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    return np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * (K @ K)


def test_config1_reference_test_on_the_facade(torch, oracle):
    """configs[0]: ContinousContactModelTest.cpp:32-214 run against the GPU-backed facade, and
    every getter compared with the oracle object."""
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModel
    rng = np.random.default_rng(42)
    st = syn.reference_test_state(rng.uniform(-1, 1, 3), rng.uniform(-1, 1, 3))
    tw, pose, null = st["twists"][0], st["poses"][0], st["null_poses"][0]
    L, Wd, k, b = syn.REFERENCE_TEST_PARAMS
    model = ContinuousContactModel()
    assert model.initialize(_handler())
    model.setState(tw, pose)
    model.setNullForceTransform(null)

    om = oracle.ContinuousContactModel()
    om.initialize({"length": L, "width": Wd, "spring_coeff": k, "damper_coeff": b})
    om.setState(tw, pose)
    om.setNullForceTransform(null)
    assert_parity(model.getContactWrench()[None], om.getContactWrench()[None], "wrench")
    assert_parity(model.getAutonomousDynamics()[None], om.getAutonomousDynamics()[None], "autodyn")
    assert_parity(model.getControlMatrix().reshape(1, 36), om.getControlMatrix().reshape(1, 36),
                  "ctrl")
    assert_parity(model.getRegressor().reshape(1, 12), om.getRegressor().reshape(1, 12),
                  "regressor")
    assert_ctrl_structure(model.getControlMatrix())

    # "Test contact wrench" (:60-104): Monte-Carlo surface integral, 1e4 samples, abs 1e-2
    samples = 10000
    xs = rng.uniform(-L / 2, L / 2, samples)
    ys = rng.uniform(-Wd / 2, Wd / 2, samples)
    f, t = model.surfacePointWrenches(xs, ys)
    num = np.concatenate([f.sum(0), t.sum(0)]) / samples * (L * Wd) * abs(pose[11])
    assert np.all(np.abs(num - model.getContactWrench()) <= 1e-2)
    # single-point getters agree with the oracle's, inside, on the boundary and outside
    for x, y in ((0.01, -0.02), (L / 2, Wd / 2), (L / 2 + 1e-9, 0.0), (0.0, -Wd)):
        np.testing.assert_allclose(model.getForceAtPoint(x, y), om.getForceAtPoint(x, y),
                                   rtol=1e-12, atol=1e-300)
        np.testing.assert_allclose(model.getTorqueGeneratedAtPoint(x, y),
                                   om.getTorqueGeneratedAtPoint(x, y), rtol=1e-12, atol=1e-300)

    # "Test regressor" (:107-124): abs 1e-7
    assert np.all(np.abs(model.getRegressor() @ np.array([k, b]) - model.getContactWrench()) <= 1e-7)

    # "Test contact dynamics" (:126-213): central difference, step 1e-6, abs 1e-4
    acc = np.ones(6)
    dt = 1e-6
    rate = model.getAutonomousDynamics() + model.getControlMatrix() @ acc
    Rm = pose[3:].reshape(3, 3)
    wr = []
    for sgn in (-1.0, 1.0):
        p = pose[:3] + sgn * tw[:3] * dt
        Rn = _rodrigues(sgn * tw[3:] * dt) @ Rm
        model.setState(tw + sgn * acc * dt, np.concatenate([p, Rn.reshape(9)]))
        model.setNullForceTransform(null)
        wr.append(model.getContactWrench().copy())
    assert np.all(np.abs((wr[1] - wr[0]) / (2 * dt) - rate) <= 1e-4)


def test_facade_lazy_flags_and_stale_coefficient_quirk(torch):
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModel
    st = syn.reference_test_state()
    m = ContinuousContactModel()
    assert m.initialize(_handler())
    m.setState(st["twists"][0], st["poses"][0])
    w0 = m.getContactWrench().copy()
    launches = m._handle.launch_count
    m.getContactWrench()
    assert m._handle.launch_count == launches          # cached: no second evaluation
    m.springCoeff = 4000.0                              # does not clear the flags (:256-274)
    assert np.array_equal(m.getContactWrench(), w0)
    m.setNullForceTransform(st["null_poses"][0])
    assert not np.array_equal(m.getContactWrench(), w0)


# --- sampling-MPC epilogue ----------------------------------------------------------------------------

@pytest.mark.parametrize("heterogeneous", [False, True])
@pytest.mark.parametrize("rollout_len,n_rollouts,mask", [(200, 512, 0), (200, 300, FULL),
                                                         (7, 1000, W), (33, 64, Cc)])
def test_rollout_cost_argmin(torch, batch, oracle, heterogeneous, rollout_len, n_rollouts, mask):
    n = rollout_len * n_rollouts
    st = syn.make_states(n, seed=31, heterogeneous=heterogeneous)
    planes, prm = _soa_inputs(torch, st)
    ref_wrench = np.array([1.0, -2.0, 30.0, 0.1, 0.2, -0.3])
    weights = np.array([1.0, 25.0])
    out, cost, best = batch.rollout_cost_argmin(planes, rollout_len, ref_wrench, weights, prm,
                                                mask=mask, index_base=1000)
    ref = oracle.eval_batch_states(st, mask=mask | W, nthreads=NTHREADS)
    ref_cost = oracle.rollout_cost(ref["wrench"], rollout_len, ref_wrench, weights)
    cost = cost.cpu().numpy()
    np.testing.assert_allclose(cost, ref_cost, rtol=1e-12)
    bc, bi = batch.decode_best(best)
    j = int(np.argmin(cost))                    # first minimum = lowest-index tie-break
    assert bi == 1000 + j and bc == cost[j]
    assert ref_cost[bi - 1000] <= ref_cost.min() * (1 + 1e-12)
    if mask:
        _check(_soa_out_to_aos(out), ref, mask, "rollout outputs")
    # determinism of the fused reduction
    _, cost2, best2 = batch.rollout_cost_argmin(planes, rollout_len, ref_wrench, weights, prm,
                                                mask=0, index_base=1000)
    assert np.array_equal(cost2.cpu().numpy(), cost) and torch.equal(best, best2)


def test_argmin_pairs_tie_break(torch, batch):
    pairs = torch.tensor([[3.0, 5], [1.5, 9], [1.5, 4], [2.0, 1]], dtype=torch.float64)
    packed = torch.empty((4, 2), dtype=torch.int64)
    packed[:, 0] = pairs[:, 0].contiguous().view(torch.int64)
    packed[:, 1] = pairs[:, 1].to(torch.int64)
    best = batch.argmin_pairs(packed.cuda())
    assert batch.decode_best(best) == (1.5, 4)


def test_config4_full_size_64m_heterogeneous_properties(torch, batch, oracle):
    """configs[3] at its full size (335 544 rollouts x 200 = 67 108 800 heterogeneous states) on one
    GPU: oracle parity on a strided sample of the same device bits, per-rollout cost on sampled
    rollouts, arg-min consistency, control-matrix structure over the whole batch."""
    free, _ = torch.cuda.mem_get_info()
    if free < 60e9:
        pytest.skip("needs ~45 GB of free device memory")
    n_rollouts, rl = 335544, 200
    n = n_rollouts * rl
    planes, prm = syn.make_planes_torch(n, torch.device("cuda", 0), seed=46, heterogeneous=True)
    ref_wrench, weights = [0.0, 0.0, 30.0, 0.0, 0.0, 0.0], [1.0, 10.0]
    out, cost, best = batch.rollout_cost_argmin(planes, rl, ref_wrench, weights, prm, mask=FULL)
    torch.cuda.synchronize()
    # (i) oracle parity on every 4099th state
    idx = torch.arange(0, n, 4099, device="cuda")
    st = syn.sample_states_from_planes(planes, prm, idx)
    ref = oracle.eval_batch_states(st, mask=FULL, nthreads=NTHREADS)
    got = {"wrench": out["wrench"][:, idx].T.cpu().numpy(), "autodyn": out["autodyn"][:, idx].T.cpu().numpy(),
           "ctrl": out["ctrl"][idx].cpu().numpy()}
    _check(got, ref, FULL, "config4 full size")
    # (ii) cost of sampled rollouts against the oracle on those rollouts' 200 states
    for r in (0, 1, 777, 200000, n_rollouts - 1):
        ridx = torch.arange(r * rl, (r + 1) * rl, device="cuda")
        rs = syn.sample_states_from_planes(planes, prm, ridx)
        rw = oracle.eval_batch_states(rs, mask=W)["wrench"]
        rc = oracle.rollout_cost(rw, rl, ref_wrench, weights)[0]
        assert abs(float(cost[r]) - rc) <= 1e-12 * abs(rc)
    # (iii) arg-min is the first minimum of the device's own cost vector
    bc, bi = batch.decode_best(best)
    j = int(torch.argmin(cost))
    cmin = float(cost[j])
    first = int(torch.nonzero(cost == cmin)[0])
    assert bi == first and bc == cmin
    # (iv) structural zeros over all 67M dense blocks, on the device
    c = out["ctrl"].view(n, 6, 6)
    assert not bool(c[:, :3, 3:].any()) and not bool(c[:, 3:, :3].any())
    offdiag = c[:, :3, :3].clone()
    offdiag.diagonal(dim1=1, dim2=2).zero_()
    assert not bool(offdiag.any())
    del offdiag
    assert bool(torch.isfinite(out["wrench"]).all()) and bool(torch.isfinite(out["autodyn"]).all())


@pytest.mark.parametrize("n", [1, 31, 33, 65, 129, 4097])
def test_no_out_of_bounds_writes_canaries(torch, batch, n):
    """compute-sanitizer is closed on this pool: every output lives between sentinel-filled guard
    bands (and inputs are followed by NaN guards, so an over-read would poison a result)."""
    guard, sentinel = 64, -7.25
    st = syn.make_states(n, seed=3, heterogeneous=True)

    def guarded(rows, cols, fill=sentinel):
        """(rows, cols) view with `guard` doubles of sentinel before and after every row."""
        buf = torch.full((rows, cols + 2 * guard), fill, dtype=torch.float64, device="cuda")
        return buf, buf[:, guard:guard + cols]

    def check(buf, cols, what):
        assert bool((buf[:, :guard] == sentinel).all()) and \
            bool((buf[:, guard + cols:] == sentinel).all()), f"{what}: guard band overwritten (n={n})"

    # SoA: planes with NaN guards after each row, outputs with sentinel guards
    pbuf = torch.full((30, n + 2 * guard), float("nan"), dtype=torch.float64, device="cuda")
    planes = pbuf[:, guard:guard + n]
    planes.copy_(_dev(torch, syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])))
    qbuf = torch.full((4, n + 2 * guard), float("nan"), dtype=torch.float64, device="cuda")
    prm = qbuf[:, guard:guard + n]
    prm.copy_(_dev(torch, st["params"].T))
    wb, w = guarded(6, n)
    ab, a = guarded(6, n)
    rb, r = guarded(12, n)
    cb, c = guarded(1, n * 36)
    out = {"wrench": w, "autodyn": a, "regressor": r, "ctrl": c.view(n, 36)}
    batch.evaluate_soa(planes, prm, FULL | R, out=out)
    torch.cuda.synchronize()
    for b_, cols, what in ((wb, n, "wrench"), (ab, n, "autodyn"), (rb, n, "regressor"),
                           (cb, n * 36, "ctrl")):
        check(b_, cols, "soa " + what)
    assert bool(torch.isfinite(w).all()) and bool(torch.isfinite(c).all())   # no NaN guard was read

    # rollout epilogue on the same guarded buffers (rollout_len 1 and n)
    for rl in (1, n):
        costb, cost = guarded(1, n // rl)
        for b_ in (wb, ab, cb):
            b_[:, guard:-guard].fill_(0.0)
        import ctypes as C
        from bipedal_locomotion_framework_b200 import _capi
        best = torch.empty(2, dtype=torch.int64, device="cuda")
        ref = np.zeros(6)
        wts = np.ones(2)
        pp = batch._plane_ptrs
        rc = _capi.lib().blf_ccm_rollout_cost_argmin_soa(
            batch.handle.ptr, n // rl, rl, pp(planes, 30), pp(prm, 4), FULL, pp(w, 6), pp(a, 6),
            c.data_ptr(), ref.ctypes.data_as(C.c_void_p), wts.ctypes.data_as(C.c_void_p), 0,
            cost.data_ptr(), best.data_ptr(), None)
        assert rc == 0, _capi.lib().blf_ccm_last_error()
        torch.cuda.synchronize()
        check(costb, n // rl, f"rollout cost rl={rl}")
        for b_, cols, what in ((wb, n, "wrench"), (ab, n, "autodyn"), (cb, n * 36, "ctrl")):
            check(b_, cols, f"rollout {what} rl={rl}")
        assert bool(torch.isfinite(cost).all())

    # AoS: each array inside guards (16-byte aligned: guard is even)
    def guarded_aos(arr, fill):
        flat = torch.full((arr.size + 2 * guard,), fill, dtype=torch.float64, device="cuda")
        v = flat[guard:guard + arr.size].view(arr.shape)
        v.copy_(torch.from_numpy(np.ascontiguousarray(arr)))
        return flat, v

    _, tw = guarded_aos(st["twists"], float("nan"))
    _, po = guarded_aos(st["poses"], float("nan"))
    _, nu = guarded_aos(st["null_poses"], float("nan"))
    _, pr = guarded_aos(st["params"], float("nan"))
    outs = {}
    flats = {}
    for key, width in (("wrench", 6), ("autodyn", 6), ("ctrl", 36), ("regressor", 12)):
        flats[key], outs[key] = guarded_aos(np.zeros((n, width)), sentinel)
    batch.evaluate_aos(tw, po, nu, pr, FULL | R, out=outs)
    torch.cuda.synchronize()
    for key, width in (("wrench", 6), ("autodyn", 6), ("ctrl", 36), ("regressor", 12)):
        f = flats[key]
        assert bool((f[:guard] == sentinel).all()) and bool((f[guard + n * width:] == sentinel).all()), \
            f"aos {key}: guard band overwritten (n={n})"
        assert bool(torch.isfinite(outs[key]).all())


# --- round 2 ------------------------------------------------------------------------------------------

def test_config5_full_size_256m_properties(torch, batch, oracle):
    """configs[4] at its full size: 2^28 states (2^20 rollouts x 256), uniform, wrench + autonomous
    dynamics + control matrix on ONE GPU (58 GB of live input planes + 103 GB of outputs): oracle
    parity on a strided sample plus the first and last 2^20 states of the same device bits,
    per-rollout cost on sampled rollouts, arg-min consistency, structural zeros over all 2^28 dense
    blocks scanned on the device."""
    import gc
    gc.collect()
    torch.cuda.empty_cache()   # blocks cached by earlier tests of this process count as used
    free, total = torch.cuda.mem_get_info()
    if free < 166e9:
        pytest.skip(f"needs ~165 GB of free device memory (free {free / 1e9:.1f} of {total / 1e9:.1f} GB)")
    n_rollouts, rl = 1 << 20, 256
    n = n_rollouts * rl
    dev = torch.device("cuda", 0)
    ref_wrench, weights = [0.0, 0.0, 30.0, 0.0, 0.0, 0.0], [1.0, 10.0]
    try:
        planes, _ = syn.make_planes_torch(n, dev, seed=46)
        out, cost, best = batch.rollout_cost_argmin(planes, rl, ref_wrench, weights, None, mask=FULL)
    except torch.cuda.OutOfMemoryError as e:   # another process took memory after the check above
        planes = out = None
        gc.collect()
        torch.cuda.empty_cache()
        pytest.skip(f"161 GB working set does not fit beside what else is on the device: {e}")
    torch.cuda.synchronize()
    # (i) oracle parity: every 4099th state (65 489 states), then the first and the last 2^20
    for what, idx in (("strided", torch.arange(0, n, 4099, device=dev)),
                      ("first 2^20", torch.arange(0, 1 << 20, device=dev)),
                      ("last 2^20", torch.arange(n - (1 << 20), n, device=dev))):
        st = syn.sample_states_from_planes(planes, None, idx)
        ref = oracle.eval_batch_states(st, mask=FULL, nthreads=NTHREADS)
        got = {"wrench": out["wrench"][:, idx].T.cpu().numpy(),
               "autodyn": out["autodyn"][:, idx].T.cpu().numpy(), "ctrl": out["ctrl"][idx].cpu().numpy()}
        _check(got, ref, FULL, f"config5 full size, {what}")
        del st, ref, got
    # (ii) cost of sampled rollouts
    for r in (0, 1, 4097, 777777, n_rollouts - 1):
        ridx = torch.arange(r * rl, (r + 1) * rl, device=dev)
        rs = syn.sample_states_from_planes(planes, None, ridx)
        rw = oracle.eval_batch_states(rs, mask=W)["wrench"]
        rc = oracle.rollout_cost(rw, rl, ref_wrench, weights)[0]
        assert abs(float(cost[r]) - rc) <= 1e-12 * abs(rc)
    # (iii) arg-min = first minimum of the device's own cost vector
    bc, bi = batch.decode_best(best)
    cmin = float(cost.min())
    assert bi == int(torch.nonzero(cost == cmin)[0]) and bc == cmin
    # (iv) structural zeros, exactly +0.0 (bit pattern 0), over all 2^28 blocks; chunked so the
    # temporaries stay under 1 GB next to the 161 GB working set
    zero_cols = torch.tensor([j for j in range(36)
                              if not ((j // 6 < 3 and j % 6 == j // 6) or (j // 6 >= 3 and j % 6 >= 3))],
                             device=dev)
    bits = out["ctrl"].view(torch.int64)
    step = 1 << 22
    for a in range(0, n, step):
        blk = bits[a:a + step]
        assert not bool(blk.index_select(1, zero_cols).any()), f"structural zero not +0.0 in block {a}"
        assert bool((blk[:, 0] == blk[:, 7]).all()) and bool((blk[:, 0] == blk[:, 14]).all())
        assert bool((blk[:, 22] == blk[:, 27]).all()) and bool((blk[:, 23] == blk[:, 33]).all()) \
            and bool((blk[:, 29] == blk[:, 34]).all())          # bottom-right block symmetric
    for p in out["wrench"]:
        assert bool(torch.isfinite(p).all())
    for p in out["autodyn"]:
        assert bool(torch.isfinite(p).all())
    del planes, out, cost, best, bits
    gc.collect()
    torch.cuda.empty_cache()   # hand the 161 GB back before the next test


@pytest.mark.parametrize("n", [2, 33, 4097, 65536, 65537, 200003])
@pytest.mark.parametrize("pinned", [False, True])
def test_host_path_compact_download_is_bit_identical_to_dense(torch, batch, oracle, n, pinned):
    """blf_ccm_eval_batch_host moves the control matrix over PCIe as its 7 distinct values and
    expands it on the host: the dense array must be bit-identical to the dense download (every
    structural zero +0.0), for ragged sizes across the chunk boundary, pageable and pinned buffers,
    and a destination that is only 8-byte aligned."""
    st = syn.make_states(n, seed=77, heterogeneous=True)
    mk = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()) if pinned else np.ascontiguousarray
    tw, po, nu, pr = mk(st["twists"]), mk(st["poses"]), mk(st["null_poses"]), mk(st["params"])
    try:
        batch.set_host_threads(0)
        dense = batch.evaluate_host(tw, po, nu, pr, FULL | R)
        for threads in (1, 3, -1):
            batch.set_host_threads(threads)
            # 8-byte-aligned (not 16) destination for the dense array on odd thread counts
            raw = np.full(n * 36 + 1, -7.25)
            ctrl = raw[1:].reshape(n, 36) if threads == 3 and raw.ctypes.data % 16 == 0 else raw[:n * 36].reshape(n, 36)
            outp = {"wrench": np.empty((n, 6)), "autodyn": np.empty((n, 6)), "ctrl": ctrl,
                    "regressor": np.empty((n, 12))}
            got = batch.evaluate_host(tw, po, nu, pr, FULL | R, out=outp)
            for key in ("wrench", "autodyn", "ctrl", "regressor"):
                assert np.array_equal(got[key].view(np.int64), dense[key].view(np.int64)), \
                    f"{key} differs, n={n}, threads={threads}"
            assert_ctrl_structure(got["ctrl"])
        # control matrix alone (no state arrays needed) and repeated calls on the same handle
        only = batch.evaluate_host(None, po, None, pr, Cc)
        assert np.array_equal(only["ctrl"].view(np.int64), dense["ctrl"].view(np.int64))
    finally:
        batch.set_host_threads(-1)
    ref = oracle.eval_batch_states(st, mask=FULL | R, nthreads=NTHREADS)
    _check(dense, ref, FULL, "host path")


def test_rollout_calls_on_two_streams_are_serialised_not_corrupted(torch, batch, oracle):
    """The rollout scratch (per-rollout partial sums, last-block counter) is one set per handle: two
    asynchronous rollout calls on DIFFERENT streams must be ordered by the library, each producing
    the result it would produce alone."""
    rl = 200
    sa, sb = syn.make_states(3000 * rl, seed=5), syn.make_states(1111 * rl, seed=6)
    pa, _ = _soa_inputs(torch, sa)
    pb, _ = _soa_inputs(torch, sb)
    ref_w, wts = [0.0, 0.0, 30.0, 0.0, 0.0, 0.0], [1.0, 10.0]
    _, ca0, ba0 = batch.rollout_cost_argmin(pa, rl, ref_w, wts)
    _, cb0, bb0 = batch.rollout_cost_argmin(pb, rl, ref_w, wts)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(20):
        with torch.cuda.stream(s1):
            _, ca, ba = batch.rollout_cost_argmin(pa, rl, ref_w, wts)
        with torch.cuda.stream(s2):
            _, cb, bb = batch.rollout_cost_argmin(pb, rl, ref_w, wts)
        torch.cuda.synchronize()
        assert torch.equal(ca, ca0) and torch.equal(cb, cb0)
        assert torch.equal(ba, ba0) and torch.equal(bb, bb0)


def test_calls_restore_the_callers_current_device(torch, batch):
    """Every C-ABI call makes the handle's device current only for its own duration."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch
    other = ContinuousContactModelBatch(1)
    other.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    st = syn.make_states(1000, seed=9)
    torch.cuda.set_device(0)
    got = other.evaluate_host(st["twists"], st["poses"], st["null_poses"], None, FULL)
    assert torch.cuda.current_device() == 0
    x = torch.zeros(4, device="cuda")          # the caller's next allocation lands on ITS device
    assert x.device.index == 0
    ref = batch.evaluate_host(st["twists"], st["poses"], st["null_poses"], None, FULL)
    for key in ("wrench", "autodyn", "ctrl"):
        assert np.array_equal(got[key], ref[key])


def test_facade_one_launch_per_state(torch, oracle):
    """The per-instance facade evaluates all four outputs with ONE launch on the first getter after
    a setter; the other getters of the same state launch nothing.  Writing springCoeff in between
    keeps the reference's quirk: results already served stay stale, results not yet computed use
    the new coefficient (src/ContactModels/src/ContinuousContactModel.cpp:256-274)."""
    from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModel, StdImplementation
    h = StdImplementation()
    for k, v in zip(("length", "width", "spring_coeff", "damper_coeff"), syn.REFERENCE_TEST_PARAMS):
        h.setParameter(k, v)
    m = ContinuousContactModel(0)
    assert m.initialize(h)
    st = syn.reference_test_state()
    m.setNullForceTransform(st["null_poses"][0])
    m.setState(st["twists"][0], st["poses"][0])
    before = m._handle.launch_count
    w = m.getContactWrench().copy()
    assert m._handle.launch_count == before + 1
    a, c, r = m.getAutonomousDynamics().copy(), m.getControlMatrix().copy(), m.getRegressor().copy()
    assert m._handle.launch_count == before + 1
    ref = oracle.eval_batch_states(st, mask=FULL | R)
    assert_parity(w[None], ref["wrench"], "wrench")
    assert_parity(a[None], ref["autodyn"], "autodyn")
    assert_parity(c.reshape(1, 36), ref["ctrl"], "ctrl")
    assert_parity(r.reshape(1, 12), ref["regressor"], "regressor")
    # stale-cache quirk through the one-launch cache
    m.setState(st["twists"][0], st["poses"][0])
    w1 = m.getContactWrench().copy()
    m.springCoeff = 2.0 * syn.REFERENCE_TEST_PARAMS[2]
    assert np.array_equal(m.getContactWrench(), w1)                    # served stale, as upstream
    a2 = m.getAutonomousDynamics().copy()                               # computed now: new coefficient
    st2 = dict(st, uniform=(syn.REFERENCE_TEST_PARAMS[0], syn.REFERENCE_TEST_PARAMS[1],
                            2.0 * syn.REFERENCE_TEST_PARAMS[2], syn.REFERENCE_TEST_PARAMS[3]))
    ref2 = oracle.eval_batch_states(st2, mask=FULL)
    assert_parity(a2[None], ref2["autodyn"], "autodyn")
    assert not np.array_equal(a2, a)
    m.setState(st["twists"][0], st["poses"][0])
    assert_parity(m.getContactWrench()[None], ref2["wrench"], "wrench")  # the next setState refreshes
