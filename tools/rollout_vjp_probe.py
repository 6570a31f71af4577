"""Throughput of the rollout cost's reverse mode (blf_ccm_rollout_cost_vjp) against the cost-only forward
rollout and the device's copy peak.

Shapes (rollouts x feet x horizon): 4 096 x 2 x 100 at rho = 0.01 and 0 (the sampling-MPC size), and
65 536 x 2 x 100 at rho = 0.01 (working set 2 x 52 MB of twists and gradients + tape, beyond L2).
Every group is requested with uniform parameters.  Each call is timed with CUDA events, median of
--reps calls after a warm-up, with tape segments of 8 steps (the default) and of 4
(BLF_CCM_TUNE_VJP_SEG=4 on a second handle).  Algorithmic bytes per chain-step: 48 (twist, forward
sweep) + 48 (twist, reverse sweep) + 48 (twist gradient) + 2 x 96 / S (tape written and read).
The FP64 instruction count per chain-step is read from the kernel's SASS (cuobjdump) when the tool is
on the PATH.  The card name and power limit are read in the same run.

  python tools/rollout_vjp_probe.py [--reps 20] [--log FILE]
"""
from __future__ import annotations

import argparse
import os
import re
import shutil
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bipedal_locomotion_framework_b200 import build  # noqa: E402
from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch  # noqa: E402
from bipedal_locomotion_framework_b200.system import RolloutBatch  # noqa: E402


def ev_time(fn, reps):
    for _ in range(3):
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


def sass_fp64_counts():
    """Static FP64 instruction counts of the all-groups kernels, uniform parameters, per (rho != 0, S)."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        return {}
    txt = subprocess.run([tool, "-sass", build.CUDA_LIB], stdout=subprocess.PIPE, text=True).stdout
    out, cur = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            k = re.match(r"_ZN6blfccm22ccm_rollout_vjp_kernelILb0ELb(\d)ELj15ELi(\d+)E", m.group(1))
            cur = (k.group(1) == "1", int(k.group(2))) if k else None
            if cur:
                out[cur] = 0
        elif cur and re.search(r"\b(DFMA|DMUL|DADD|MUFU\.RCP64H)\b", line):
            out[cur] += 1
    return out


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
                          "--format=csv", "-i", "0"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    for ln in smi.stdout.strip().splitlines():
        log(ln)
    dev = torch.device("cuda", 0)
    log(f"device: {torch.cuda.get_device_name(dev)}, torch {torch.__version__}, CUDA {torch.version.cuda}")
    fp64 = sass_fp64_counts()
    for (baum, s), n in sorted(fp64.items()):
        log(f"SASS: all-groups kernel, rho {'!= 0' if baum else '== 0'}, S = {s}: {n} FP64 instructions (static)")

    src = torch.empty(1 << 29, dtype=torch.float64, device=dev).fill_(1.0)
    dst = torch.empty_like(src)
    med, lo, hi = ev_time(lambda: dst.copy_(src), args.reps)
    peak = 2 * src.numel() * 8 / med
    log(f"d2d copy 4 GiB: median {med * 1e3:.3f} ms (min {lo * 1e3:.3f}, max {hi * 1e3:.3f}) -> {peak / 1e9:.0f} GB/s")
    del src, dst

    import rollout_grad_reference as ref
    rbs = {}
    for seg in (8, 4):
        os.environ["BLF_CCM_TUNE_VJP_SEG"] = str(seg)
        b = ContinuousContactModelBatch(0)
        b.set_uniform_params(0.2, 0.1, 1e6, 1e4)
        rbs[seg] = RolloutBatch(b)
    os.environ.pop("BLF_CCM_TUNE_VJP_SEG")
    for nr, feet, H, rho in ((4096, 2, 100, 0.01), (4096, 2, 100, 0.0), (65536, 2, 100, 0.01)):
        case = ref.make_case(nr, feet, H, seed=1)
        d = {k: torch.from_numpy(case[k]).to(dev) for k in ("twist", "pos", "rot", "null")}
        a = (nr, feet, H, 0.01, rho, d["twist"], d["pos"], d["rot"], d["null"], ref.REF, ref.WEIGHTS)
        gcost = torch.ones(nr, dtype=torch.float64, device=dev)
        fwd, _ = rbs[8].prepare(*a)
        f_med, _, _ = ev_time(fwd, args.reps)
        cs = nr * feet * H
        log(f"{nr} x {feet} x {H}, rho {rho}: forward cost-only rollout median {f_med * 1e6:9.1f} us "
            f"({cs / f_med / 1e9:6.2f} G chain-steps/s)")
        for seg in (8, 4):
            call, _ = rbs[seg].prepare_cost_vjp(*a, gcost)
            med, lo, hi = ev_time(call, args.reps)
            bps = 144 + 192 / seg
            n64 = fp64.get((rho != 0.0, seg))
            log(f"  VJP all groups, S = {seg}: median {med * 1e6:9.1f} us (min {lo * 1e6:.1f}, max {hi * 1e6:.1f})  "
                f"{cs / med / 1e9:6.2f} G chain-steps/s  = {med / f_med:5.2f} x forward  "
                f"{bps:.0f} B/chain-step -> {cs * bps / med / 1e9:6.0f} GB/s = {cs * bps / med / peak:.3f} of the copy peak"
                + (f"  ~{n64} FP64 instr/chain-step (static) -> {cs * n64 / 32 / med / 148 / 1e9:.2f} G warp-instr/s/SM"
                   if n64 else ""))
        del d, case
        torch.cuda.empty_cache()
    if args.log:
        os.makedirs(os.path.dirname(os.path.abspath(args.log)), exist_ok=True)
        with open(args.log, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
