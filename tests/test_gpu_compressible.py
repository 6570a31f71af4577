"""The dense control-matrix outputs in compressible device memory (blf_ccm_device_alloc_compressible).

Compression happens between L2 and HBM and must be invisible: every output written into a
compressible ctrl array is bit-identical to the same call into plain torch.empty memory, the structural
zeros stay exact +0.0, memory next to the array is untouched, and the allocation lives as long as any
view of it and is released only after the work that uses it."""
import ctypes as C

import numpy as np
import pytest

from bipedal_locomotion_framework_b200 import _capi
from bipedal_locomotion_framework_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

FULL = 7
REF, WTS = [0.0, 0.0, 30.0, 0.0, 0.0, 0.0], [1.0, 10.0]
ROLLOUT_LEN = 200
N_ROLLOUTS = 5243                  # 1 048 600 = 2^20 + 24 states: the last warp tile is ragged
ZMASK = np.ones(36, dtype=bool)
for _q in range(3):
    ZMASK[6 * _q + _q] = False
    ZMASK[6 * (3 + _q) + 3: 6 * (3 + _q) + 6] = False


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
def supported():
    """CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED of device 0, from the driver."""
    cu = C.CDLL("libcuda.so.1")
    v = C.c_int()
    assert cu.cuDeviceGetAttribute(C.byref(v), C.c_int(107), C.c_int(0)) == 0
    return bool(v.value)


@pytest.fixture(scope="module")
def planes(torch):
    pl, _ = syn.make_planes_torch(N_ROLLOUTS * ROLLOUT_LEN, torch.device("cuda", 0), seed=46)
    return pl


@pytest.fixture(scope="module")
def plain_ref(torch, batch, planes, monkeypatch_module):
    """The headline call into plain torch.empty outputs."""
    monkeypatch_module.setenv("BLF_CCM_TUNE_NO_COMPRESS", "1")
    out, cost, best = batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL)
    monkeypatch_module.delenv("BLF_CCM_TUNE_NO_COMPRESS")
    torch.cuda.synchronize()
    assert batch.handle.last_path == _capi.PATH_BULK
    assert not batch.is_compressible(out["ctrl"])
    return out, cost, best


@pytest.fixture(scope="module")
def monkeypatch_module():
    mp = pytest.MonkeyPatch()
    yield mp
    mp.undo()


def _ptr_is_compressible(batch, ptr: int) -> bool:
    out = C.c_int()
    _capi.check(_capi.lib().blf_ccm_pointer_is_compressible(batch.handle.ptr, ptr, C.byref(out)))
    return bool(out.value)


def _zeros_exact(torch, ctrl) -> bool:
    cols = torch.from_numpy(np.nonzero(ZMASK)[0]).to(ctrl.device)
    return bool((ctrl.index_select(1, cols).view(torch.int64) == 0).all())


def _assert_same(torch, a, b):
    (oa, ca, ba), (ob, cb, bb) = a, b
    for k in ("wrench", "autodyn", "ctrl"):
        assert torch.equal(oa[k], ob[k]), k
    assert torch.equal(ca, cb)
    assert torch.equal(ba, bb)


def test_ctrl_is_compressible_where_supported(torch, batch, supported, monkeypatch):
    out = batch.alloc_soa_outputs(4096, FULL)
    assert batch.is_compressible(out["ctrl"]) == supported
    assert batch.is_compressible(out["ctrl"][100:]) == supported
    assert not batch.is_compressible(out["wrench"])
    assert batch.is_compressible(batch.alloc_aos_outputs(4096, FULL)["ctrl"]) == supported
    monkeypatch.setenv("BLF_CCM_TUNE_NO_COMPRESS", "1")
    assert not batch.is_compressible(batch.alloc_soa_outputs(4096, FULL)["ctrl"])
    assert not batch.is_compressible(batch.alloc_aos_outputs(4096, FULL)["ctrl"])
    assert batch.alloc_soa_outputs(0, FULL)["ctrl"].shape == (0, 36)


def test_rollout_bit_identical_bulk_path(torch, batch, planes, plain_ref, supported):
    out = batch.alloc_soa_outputs(N_ROLLOUTS * ROLLOUT_LEN, FULL)
    assert batch.is_compressible(out["ctrl"]) == supported
    got = batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL, out=out)
    torch.cuda.synchronize()
    assert batch.handle.last_path == _capi.PATH_BULK
    _assert_same(torch, got, plain_ref)
    assert _zeros_exact(torch, got[0]["ctrl"])


def test_rollout_bit_identical_misaligned_path(torch, batch, planes, plain_ref, supported):
    """ctrl 8 bytes past a 16-byte boundary: the kernel's direct 64-bit store path."""
    n = N_ROLLOUTS * ROLLOUT_LEN
    base = batch.alloc_ctrl(n + 1)
    assert batch.is_compressible(base) == supported
    out = batch.alloc_soa_outputs(n, FULL & ~4)
    out["ctrl"] = base.view(-1)[1: 1 + 36 * n].view(n, 36)
    got = batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL, out=out)
    torch.cuda.synchronize()
    assert batch.handle.last_path == _capi.PATH_DIRECT64
    _assert_same(torch, got, plain_ref)
    assert _zeros_exact(torch, got[0]["ctrl"])


def test_aos_and_host_paths_into_compressible_ctrl(torch, batch, monkeypatch):
    n = 100_003
    st = syn.make_states(n, seed=11)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    tw, po, nu = dev(st["twists"]), dev(st["poses"]), dev(st["null_poses"])
    got = batch.evaluate_aos(tw, po, nu, mask=FULL)
    torch.cuda.synchronize()
    monkeypatch.setenv("BLF_CCM_TUNE_NO_COMPRESS", "1")
    ref = batch.evaluate_aos(tw, po, nu, mask=FULL)
    torch.cuda.synchronize()
    host = batch.evaluate_host(st["twists"], st["poses"], st["null_poses"], mask=FULL)
    for k in ("wrench", "autodyn", "ctrl"):
        assert torch.equal(got[k], ref[k]), k
        assert np.array_equal(got[k].cpu().numpy(), host[k]), k
    assert _zeros_exact(torch, got["ctrl"])


def test_lifetime_views_and_pending_work(torch, batch, planes, plain_ref, supported):
    n = N_ROLLOUTS * ROLLOUT_LEN
    ref_ctrl = plain_ref[0]["ctrl"]
    out = batch.alloc_soa_outputs(n, FULL)
    batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL, out=out)
    keep = out["ctrl"][n - 5000: n - 1000]      # a slice outlives the dict and the array
    ptr = out["ctrl"].data_ptr()
    del out
    torch.cuda.synchronize()
    assert torch.equal(keep, ref_ctrl[n - 5000: n - 1000])
    assert _ptr_is_compressible(batch, ptr) == supported
    # launch, then drop every reference with the kernel still queued: the free waits for it
    out = batch.alloc_soa_outputs(n, FULL)
    batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL, out=out)
    ptr2 = out["ctrl"].data_ptr()
    del out
    assert not _ptr_is_compressible(batch, ptr2)
    out = batch.alloc_soa_outputs(n, FULL)
    got = batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL, out=out)
    torch.cuda.synchronize()
    _assert_same(torch, got, plain_ref)
    assert torch.equal(keep, ref_ctrl[n - 5000: n - 1000])
    del keep
    assert not _ptr_is_compressible(batch, ptr)


def test_guard_bands_around_compressible_ctrl(torch, batch, planes, plain_ref):
    n, g = N_ROLLOUTS * ROLLOUT_LEN, 1024
    canary = 0x7FF8DEADBEEF0001              # a NaN bit pattern no output can have
    base = batch.alloc_ctrl(n + 2 * g)
    base.view(torch.int64).fill_(canary)
    out = batch.alloc_soa_outputs(n, FULL & ~4)
    out["ctrl"] = base[g: g + n]
    got = batch.rollout_cost_argmin(planes, ROLLOUT_LEN, REF, WTS, mask=FULL, out=out)
    torch.cuda.synchronize()
    want = torch.full((g, 36), canary, dtype=torch.int64, device=base.device)
    assert torch.equal(base[:g].view(torch.int64), want)
    assert torch.equal(base[g + n:].view(torch.int64), want)
    _assert_same(torch, got, plain_ref)
