#!/usr/bin/env python
"""Does the B200 compress the dense 6x6 control-matrix output (24 of 36 entries +0.0), and does it
make the headline step faster?  One run answers it:

  1. the device's compression attribute, the granularity of a compressible allocation, and what the
     driver actually granted for a headline-sized (2^28 x 288 B) compressible allocation;
  2. calibration: a fill of zeros, of one control-matrix row repeated, and of random doubles, each
     into 8 GB of compressible and of plain memory;
  3. the headline step exactly as bench.py binds it (2^20 rollouts x 256, FULL, uniform, cost +
     arg-min) with the ctrl array from torch.empty (arm A) or from compressible memory (arm B),
     alternated over ROUNDS rounds of STEPS steps, median and spread per arm;
  4. A and B outputs compared bit for bit: the whole of every output at 2^24 states + a ragged
     rollout, chunked 64-bit digests of every output at the headline size, and the structural zeros
     checked to be +0.0 by their bit pattern.

   python tools/compress_probe.py [--rounds 10] [--steps 20] [--log-states 28]

The driver API is reached through ctypes on libcuda (VMM: cuMemCreate / cuMemMap); the buffers are
handed to torch through __cuda_array_interface__."""
from __future__ import annotations

import argparse
import ctypes as C
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bipedal_locomotion_framework_b200 import synthetic as syn  # noqa: E402
from bipedal_locomotion_framework_b200.contact_models import FULL, ContinuousContactModelBatch  # noqa: E402

ATTR_GENERIC_COMPRESSION_SUPPORTED = 107
COMP_GENERIC = 1
GRAN_MINIMUM, GRAN_RECOMMENDED = 0, 1
REF_WRENCH, WEIGHTS = [0.0, 0.0, 30.0, 0.0, 0.0, 0.0], [1.0, 10.0]


class _Loc(C.Structure):
    _fields_ = [("type", C.c_int), ("id", C.c_int)]


class _Flags(C.Structure):
    _fields_ = [("compressionType", C.c_ubyte), ("gpuDirectRDMACapable", C.c_ubyte),
                ("usage", C.c_ushort), ("reserved", C.c_ubyte * 4)]


class _Prop(C.Structure):
    _fields_ = [("type", C.c_int), ("requestedHandleTypes", C.c_int), ("location", _Loc),
                ("win32HandleMetaData", C.c_void_p), ("allocFlags", _Flags)]


class _Access(C.Structure):
    _fields_ = [("location", _Loc), ("flags", C.c_int)]


class Driver:
    def __init__(self, device: int):
        self.cu = C.CDLL("libcuda.so.1")
        self.device = device

    def ck(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed: CUresult {rc}")

    def prop(self, compress: bool) -> _Prop:
        p = _Prop()
        p.type = 1                              # CU_MEM_ALLOCATION_TYPE_PINNED
        p.location.type, p.location.id = 1, self.device   # CU_MEM_LOCATION_TYPE_DEVICE
        p.allocFlags.compressionType = COMP_GENERIC if compress else 0
        return p

    def attribute(self, attr: int) -> int:
        v = C.c_int()
        self.ck(self.cu.cuDeviceGetAttribute(C.byref(v), C.c_int(attr), C.c_int(self.device)),
                "cuDeviceGetAttribute")
        return v.value

    def granularity(self, compress: bool, option: int) -> int:
        g = C.c_size_t()
        p = self.prop(compress)
        self.ck(self.cu.cuMemGetAllocationGranularity(C.byref(g), C.byref(p), C.c_int(option)),
                "cuMemGetAllocationGranularity")
        return g.value


class VmmBuffer:
    """One cuMemCreate allocation mapped read-write on the device; freed (after a device
    synchronise) when the last reference, e.g. a tensor made from it, goes away."""

    def __init__(self, drv: Driver, nbytes: int, compress: bool, shape, typestr="<f8"):
        self.drv, self.ptr, self.handle = drv, 0, None
        gran = drv.granularity(compress, GRAN_RECOMMENDED)
        self.size = (nbytes + gran - 1) // gran * gran
        cu = drv.cu
        p = drv.prop(compress)
        h = C.c_uint64()
        drv.ck(cu.cuMemCreate(C.byref(h), C.c_size_t(self.size), C.byref(p), C.c_ulonglong(0)), "cuMemCreate")
        self.handle = h
        got = _Prop()
        drv.ck(cu.cuMemGetAllocationPropertiesFromHandle(C.byref(got), h), "cuMemGetAllocationPropertiesFromHandle")
        self.granted = int(got.allocFlags.compressionType)
        d = C.c_uint64()
        drv.ck(cu.cuMemAddressReserve(C.byref(d), C.c_size_t(self.size), C.c_size_t(gran), C.c_uint64(0),
                                      C.c_ulonglong(0)), "cuMemAddressReserve")
        self.ptr = d.value
        drv.ck(cu.cuMemMap(C.c_uint64(self.ptr), C.c_size_t(self.size), C.c_size_t(0), h, C.c_ulonglong(0)),
               "cuMemMap")
        a = _Access()
        a.location.type, a.location.id, a.flags = 1, drv.device, 3   # CU_MEM_ACCESS_FLAGS_PROT_READWRITE
        drv.ck(cu.cuMemSetAccess(C.c_uint64(self.ptr), C.c_size_t(self.size), C.byref(a), C.c_size_t(1)),
               "cuMemSetAccess")
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr,
                                         "data": (self.ptr, False), "version": 3, "strides": None}

    def __del__(self):
        cu = self.drv.cu
        torch.cuda.synchronize()
        if self.ptr:
            cu.cuMemUnmap(C.c_uint64(self.ptr), C.c_size_t(self.size))
            cu.cuMemAddressFree(C.c_uint64(self.ptr), C.c_size_t(self.size))
        if self.handle is not None:
            cu.cuMemRelease(self.handle)


def vmm_tensor(drv, shape, compress=True):
    nbytes = int(np.prod(shape)) * 8
    buf = VmmBuffer(drv, nbytes, compress, shape)
    t = torch.as_tensor(buf, device=torch.device("cuda", drv.device))
    assert t.data_ptr() == buf.ptr
    return t, buf.granted


def ev_time(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def spread(ts):
    m = statistics.median(ts)
    return {"median_ms": m, "min_ms": min(ts), "max_ms": max(ts), "spread": (max(ts) - min(ts)) / m}


ZMASK = np.ones(36, dtype=bool)
for _q in range(3):
    ZMASK[6 * _q + _q] = False
    ZMASK[6 * (3 + _q) + 3: 6 * (3 + _q) + 6] = False
ZCOLS = torch.from_numpy(np.nonzero(ZMASK)[0])


def digest(t: torch.Tensor, chunk_bytes=1 << 30):
    """Two wrapping 64-bit digests (sum, sum of squares) of a float64 tensor's bits, per chunk."""
    v = t.reshape(-1).view(torch.int64)
    step = chunk_bytes // 8
    out = []
    for a in range(0, v.numel(), step):
        c = v[a: a + step]
        out.append((int(c.sum()), int((c * c).sum())))
    return out


def zeros_exact(ctrl: torch.Tensor, rows=1 << 22) -> bool:
    cols = ZCOLS.to(ctrl.device)
    for a in range(0, ctrl.shape[0], rows):
        if not bool((ctrl[a: a + rows].index_select(1, cols).view(torch.int64) == 0).all()):
            return False
    return True


def calibrate(drv, dev, log):
    n = (8 << 30) // 8
    row = torch.zeros(36, dtype=torch.float64, device=dev)
    row[~torch.from_numpy(ZMASK).to(dev)] = torch.tensor(
        [-2000.0, -2000.0, -2000.0, -1.5, 0.3, -0.2, -1.5, 0.3, -0.2, 0.4, 0.1, -1.5], dtype=torch.float64,
        device=dev)
    res = {}
    for kind in ("plain", "compressible"):
        if kind == "plain":
            buf, granted = torch.empty(n, dtype=torch.float64, device=dev), None
        else:
            buf, granted = vmm_tensor(drv, (n,), True)
        m = buf[: n // 36 * 36].view(-1, 36)
        fills = {"zeros": lambda: buf.zero_(),
                 "ctrl_row_repeated": lambda: m.copy_(row.expand_as(m)),
                 "random_doubles": lambda: buf.uniform_(-1.0, 1.0)}
        for name, fn in fills.items():
            fn()
            torch.cuda.synchronize()
            ts = ev_time(fn, 30)
            s = spread(ts)
            s["GB_per_s"] = (8 << 30) / (s["median_ms"] * 1e-3) / 1e9
            res[(kind, name)] = s
            log(f"calib {kind:12s} {name:18s} granted={granted} median {s['median_ms']:.3f} ms "
                f"({s['GB_per_s']:.0f} GB/s)  min {s['min_ms']:.3f} max {s['max_ms']:.3f}")
        del buf, m, fills
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    for name in ("zeros", "ctrl_row_repeated", "random_doubles"):
        log(f"calib ratio plain/compressible {name:18s} "
            f"{res[('plain', name)]['median_ms'] / res[('compressible', name)]['median_ms']:.3f}")


def headline(drv, dev, batch, log, log_states, rounds, steps, warm):
    n_roll = 1 << (log_states - 8)
    n = n_roll * 256
    planes, _ = syn.make_planes_torch(n, dev, seed=46)
    wrench = torch.empty((6, n), dtype=torch.float64, device=dev)
    autodyn = torch.empty((6, n), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    log(f"headline: {n} states ({n_roll} rollouts x 256); planes + wrench/autodyn resident; "
        f"free {torch.cuda.mem_get_info(dev)[0] / 1e9:.1f} GB before ctrl")

    def arm(kind):
        if kind == "A":
            ctrl, granted = torch.empty((n, 36), dtype=torch.float64, device=dev), None
        else:
            ctrl, granted = vmm_tensor(drv, (n, 36), True)
        out = {"wrench": wrench, "autodyn": autodyn, "ctrl": ctrl, "regressor": None}
        call, out, cost, best = batch.prepare_rollout(planes, 256, REF_WRENCH, WEIGHTS, mask=FULL, out=out)
        return call, ctrl, cost, best, granted

    med = {"A": [], "B": []}
    free_with_ctrl = {}
    last = {}
    for r in range(rounds):
        for kind in ("A", "B") if r % 2 == 0 else ("B", "A"):
            call, ctrl, cost, best, granted = arm(kind)
            free_with_ctrl[kind] = torch.cuda.mem_get_info(dev)[0]
            for _ in range(warm):
                call()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                call()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / steps
            med[kind].append(ms)
            log(f"round {r} arm {kind} granted={granted} {ms:.3f} ms/step")
            if r == rounds - 1:
                last[kind] = {"wrench": digest(wrench), "autodyn": digest(autodyn), "ctrl": digest(ctrl),
                              "cost": cost.clone(), "best": best.clone(), "zeros": zeros_exact(ctrl)}
            del call, ctrl, cost, best
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
    sa, sb = spread(med["A"]), spread(med["B"])
    log(f"arm A (torch.empty ctrl)  : median {sa['median_ms']:.3f} ms  min {sa['min_ms']:.3f} max {sa['max_ms']:.3f}"
        f"  spread {100 * sa['spread']:.2f} %")
    log(f"arm B (compressible ctrl): median {sb['median_ms']:.3f} ms  min {sb['min_ms']:.3f} max {sb['max_ms']:.3f}"
        f"  spread {100 * sb['spread']:.2f} %")
    log(f"gain A/B = {sa['median_ms'] / sb['median_ms']:.4f}")
    log(f"free memory with ctrl allocated: A {free_with_ctrl['A'] / 1e9:.2f} GB, B {free_with_ctrl['B'] / 1e9:.2f} GB")
    a, b = last["A"], last["B"]
    for k in ("wrench", "autodyn", "ctrl"):
        log(f"headline digest equal {k}: {a[k] == b[k]} ({len(a[k])} chunks)")
    log(f"headline cost equal: {torch.equal(a['cost'], b['cost'])}  best equal: {torch.equal(a['best'], b['best'])}")
    log(f"headline structural zeros exact +0.0: A {a['zeros']} B {b['zeros']}")
    del planes, wrench, autodyn
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def exact_compare(drv, dev, batch, log):
    """Whole outputs, both arms resident: 2^24 states + one more rollout (ragged for the kernel's
    tiles), then a misaligned ctrl pointer (the kernel's per-lane fallback path)."""
    n_roll = (1 << 16) + 1
    n = n_roll * 256
    planes, _ = syn.make_planes_torch(n, dev, seed=46)
    outs = {}
    for kind in ("A", "B", "B_misaligned"):
        wrench = torch.empty((6, n), dtype=torch.float64, device=dev)
        autodyn = torch.empty((6, n), dtype=torch.float64, device=dev)
        if kind == "A":
            ctrl = torch.empty((n, 36), dtype=torch.float64, device=dev)
        else:
            base, granted = vmm_tensor(drv, (n + 1, 36), True)
            ctrl = base.view(-1)[1: 1 + 36 * n].view(n, 36) if kind == "B_misaligned" else base[:n]
        out = {"wrench": wrench, "autodyn": autodyn, "ctrl": ctrl, "regressor": None}
        out, cost, best = batch.rollout_cost_argmin(planes, 256, REF_WRENCH, WEIGHTS, mask=FULL, out=out)
        torch.cuda.synchronize()
        outs[kind] = (out, cost, best, batch.handle.last_path)
    a = outs["A"]
    for kind in ("B", "B_misaligned"):
        b = outs[kind]
        eq = {k: torch.equal(a[0][k], b[0][k]) for k in ("wrench", "autodyn", "ctrl")}
        eq["cost"] = torch.equal(a[1], b[1])
        eq["best"] = torch.equal(a[2], b[2])
        log(f"exact compare A vs {kind} at {n} states (path A {a[3]}, {kind} {b[3]}): {eq}  "
            f"zeros exact: {zeros_exact(b[0]['ctrl'])}")
    del outs, a, planes
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--log-states", type=int, default=28)
    args = ap.parse_args()
    t0 = time.perf_counter()

    def log(s):
        print(f"[{time.perf_counter() - t0:7.1f}s] {s}", flush=True)

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.empty(1, device=dev)
    log(f"device: {torch.cuda.get_device_name(dev)}, torch {torch.__version__}, CUDA {torch.version.cuda}")
    drv = Driver(0)
    log(f"CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = {drv.attribute(ATTR_GENERIC_COMPRESSION_SUPPORTED)}")
    for comp in (False, True):
        log(f"granularity compress={comp}: minimum {drv.granularity(comp, GRAN_MINIMUM)} "
            f"recommended {drv.granularity(comp, GRAN_RECOMMENDED)}")
    n_head = 1 << args.log_states
    free0 = torch.cuda.mem_get_info(dev)[0]
    t, granted = vmm_tensor(drv, (n_head, 36), True)
    free1 = torch.cuda.mem_get_info(dev)[0]
    log(f"headline-sized ctrl allocation {n_head * 288 / 1e9:.1f} GB: granted compressionType = {granted}; "
        f"free memory dropped by {(free0 - free1) / 1e9:.3f} GB")
    del t
    torch.cuda.synchronize()

    batch = ContinuousContactModelBatch(0)
    batch.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    calibrate(drv, dev, log)
    exact_compare(drv, dev, batch, log)
    headline(drv, dev, batch, log, args.log_states, args.rounds, args.steps, args.warm)
    log("done")


if __name__ == "__main__":
    main()
