"""Throughput of the wrench's reverse mode (blf_ccm_wrench_vjp_soa) against the device's copy peak.

For 2^24 and 2^26 contacts it times, with CUDA events, three variants:
  all groups, uniform parameters        25 + 6 planes in, 25 + 4 out   480 B per contact
  all groups, per-contact parameters    + 4 parameter planes in        512 B per contact
  twist only                            7 + 6 in (R22, e1, e2, cotangent), 6 out   152 B per contact
Bytes are the algorithmic ones: every plane read or written once; the five structurally zero
gradient planes are passed as NULL, so they are neither counted nor written.  In the same run it
measures a device-to-device copy of 4 GiB (read + write bytes) as the practical HBM peak, and prints
the card name and power limit.  Every working set is far larger than L2.

  python tools/wrench_vjp_probe.py [--reps 20] [--log FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bipedal_locomotion_framework_b200 import _capi  # noqa: E402
from bipedal_locomotion_framework_b200 import synthetic as syn  # noqa: E402
from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch  # noqa: E402

DEAD = (11, 14, 23, 26, 29)
TWIST_READS = (9, 10, 12, 13, 15, 16, 17)


def ev_time(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def arr(ts):
    return (C.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--log", default=None)
    args = ap.parse_args()
    lines = []
    t0 = time.time()

    def log(s):
        s = f"[{time.time() - t0:7.1f}s] {s}"
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                          "--format=csv", "-i", "0"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         text=True)
    for ln in smi.stdout.strip().splitlines():
        log(ln)
    dev = torch.device("cuda", 0)
    log(f"device: {torch.cuda.get_device_name(dev)}, torch {torch.__version__}, CUDA {torch.version.cuda}")

    # practical peak: device-to-device copy, read + write bytes
    src = torch.empty(1 << 29, dtype=torch.float64, device=dev).fill_(1.0)
    dst = torch.empty_like(src)
    med, lo, hi = ev_time(lambda: dst.copy_(src), args.reps)
    peak = 2 * src.numel() * 8 / med
    log(f"d2d copy 4 GiB: median {med * 1e3:.3f} ms (min {lo * 1e3:.3f}, max {hi * 1e3:.3f}) -> {peak / 1e9:.0f} GB/s")
    del src, dst

    batch = ContinuousContactModelBatch(0)
    batch.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    fn = _capi.lib().blf_ccm_wrench_vjp_soa
    h = batch.handle.ptr
    for logn in (24, 26):
        n = 1 << logn
        planes, prm = syn.make_planes_torch(n, dev, seed=5, heterogeneous=True)
        g = torch.empty((6, n), dtype=torch.float64, device=dev).uniform_(-1.0, 1.0)
        gin = [None if i in DEAD else torch.empty(n, dtype=torch.float64, device=dev) for i in range(30)]
        gprm = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(4)]
        twist_in = [planes[i] if i in TWIST_READS else None for i in range(30)]
        twist_out = [gin[i] if i < 6 else None for i in range(30)]
        st = torch.cuda.current_stream(dev).cuda_stream
        variants = [
            ("all groups, uniform", 480, (h, n, arr(planes), None, arr(list(g)), arr(gin), arr(gprm), st)),
            ("all groups, heterogeneous", 512, (h, n, arr(planes), arr(prm), arr(list(g)), arr(gin), arr(gprm), st)),
            ("twist only, uniform", 152, (h, n, arr(twist_in), None, arr(list(g)), arr(twist_out), None, st)),
        ]
        for name, bpc, a in variants:
            def call(a=a):
                rc = fn(*a)
                if rc:
                    _capi.check(rc)
            med, lo, hi = ev_time(call, args.reps)
            bw = n * bpc / med
            log(f"n=2^{logn} {name:27s} {bpc:3d} B/contact: median {med * 1e3:8.3f} ms "
                f"(min {lo * 1e3:.3f}, max {hi * 1e3:.3f})  {bw / 1e9:6.0f} GB/s  = {bw / peak:.3f} of the copy peak")
        del planes, prm, g, gin, gprm, twist_in, twist_out
        torch.cuda.empty_cache()
    if args.log:
        os.makedirs(os.path.dirname(os.path.abspath(args.log)), exist_ok=True)
        with open(args.log, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
