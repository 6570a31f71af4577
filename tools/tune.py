#!/usr/bin/env python
"""Sweep kernel variants / launch shapes on one GPU and print a table (development aid, not the
bench).  Each row: GB/s of algorithmic bytes and fraction of the measured HBM peak."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from bipedal_locomotion_framework_b200 import synthetic as syn
from bipedal_locomotion_framework_b200.contact_models import (FULL, WRENCH,
                                                               ContinuousContactModelBatch)

try:
    PEAK = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    PEAK = 6650.0


def timeit(fn, iters=200, warm=10):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def row(name, ms, n, bytes_per):
    gbs = n * bytes_per / (ms * 1e-3) / 1e9
    print(f"{name:58s} {ms*1e3:9.1f} us  {n/ms/1e6:8.2f} G evals/s  {gbs:8.1f} GB/s  {gbs/PEAK*100:5.1f} %",
          flush=True)


def make_batch(**env):
    for k, v in env.items():
        os.environ[k] = str(v)
    b = ContinuousContactModelBatch(0)
    b.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
    return b


def rls_only():
    from bipedal_locomotion_framework_b200.estimators import RecursiveLeastSquareBatch
    b = make_batch()
    for n in (2 * 4096 * 100, 1 << 23):
        st = syn.make_states(min(n, 1 << 20), seed=45)
        reps = (n + st["n"] - 1) // st["n"]
        pl = np.tile(syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]), (1, reps))[:, :n]
        planes = torch.from_numpy(np.ascontiguousarray(pl)).cuda()
        rls = RecursiveLeastSquareBatch(b, [1.0, 1.0, 1.0, 0.01, 0.01, 0.01], 0.99)
        th = torch.rand((2, n), dtype=torch.float64, device="cuda") * 1e3 + 10
        P = torch.zeros((4, n), dtype=torch.float64, device="cuda"); P[0] = 1e6; P[3] = 1e4
        zz = torch.randn((6, n), dtype=torch.float64, device="cuda")
        Yp = torch.randn((12, n), dtype=torch.float64, device="cuda") * 1e-2
        print(f"=== n = {n} ===")
        # pre-bound calls (the Python wrappers cost more than a small launch) and, at the small
        # size, two rotating buffer sets so that a step never finds its data in the 126 MB L2
        nsets = 2 if n < (1 << 22) else 1
        sets = [(Yp.clone(), zz.clone(), th.clone(), P.clone(), planes.clone()) for _ in range(nsets)]
        calls = [rls.prepare_advance(s_[0], s_[1], s_[2], s_[3]) for s_ in sets]
        ms = timeit(lambda i: calls[i % nsets](), iters=100)
        row("rls advance p=2 m=6 (regressor planes in)", ms, n, 240)
        for s_ in sets:
            s_[3].zero_(); s_[3][0] = 1e6; s_[3][3] = 1e4
        calls = [rls.prepare_advance_contacts(s_[4], s_[1], s_[2], s_[3]) for s_ in sets]
        ms = timeit(lambda i: calls[i % nsets](), iters=100)
        row("rls fused contact identification (state planes in)", ms, n, 344)
        outs = [b.alloc_soa_outputs(n, 8) for _ in range(nsets)]
        calls = [b.prepare_soa(s_[4], None, 8, out=o)[0] for s_, o in zip(sets, outs)]
        ms = timeit(lambda i: calls[i % nsets](), iters=100)
        row("regressor-only kernel (25 planes in, 12 out)", ms, n, 296)
        del planes, th, P, zz, Yp, outs, sets, calls


def sys_only():
    """Rows 2 and 3 of SURVEY.md section 8(f): Euler step, fused rollout, J^T wrench."""
    from bipedal_locomotion_framework_b200.system import (GeneralizedForceBatch, KinematicsBatch,
                                                          RolloutBatch)
    b = make_batch()
    kb, rb, gf = KinematicsBatch(0, b.handle), RolloutBatch(b), GeneralizedForceBatch(b)
    rnd = lambda *s: torch.rand(s, dtype=torch.float64, device="cuda") * 2 - 1
    print(f"peak {PEAK} GB/s")
    # --- Euler step --------------------------------------------------------------------------------
    for n in (819200, 1 << 23):
        st = syn.make_states(min(n, 1 << 18), seed=47)
        reps = (n + st["n"] - 1) // st["n"]
        rot = torch.from_numpy(np.ascontiguousarray(np.tile(st["poses"][:, 3:].T, (1, reps))[:, :n])).cuda()
        sets = [(rnd(6, n), rnd(3, n), rot.clone()) for _ in range(3)]
        for rho in (0.0, 2.0):
            cl = [kb.prepare_euler_step(rho, 1e-4, *s_) for s_ in sets]
            ms = timeit(lambda i: cl[i % 3](), iters=100)
            row(f"kinematics euler step n={n} rho={rho}", ms, n, 240)
        del sets, rot
    # --- fused rollout -----------------------------------------------------------------------------
    for nr, feet, H in ((4096, 2, 100), (65536, 2, 100), (335544, 1, 200)):
        chains, n = nr * feet, nr * feet * H
        st = syn.make_states(min(chains, 1 << 18), seed=48)
        reps = (chains + st["n"] - 1) // st["n"]
        tile = lambda a: torch.from_numpy(np.ascontiguousarray(np.tile(a.T, (1, reps))[:, :chains])).cuda()
        pos, rot, null = tile(st["poses"][:, :3]), tile(st["poses"][:, 3:]), tile(st["null_poses"])
        tws = [rnd(6, n) for _ in range(2)]
        print(f"=== rollout {nr} x {feet} x {H} = {n} evals ===")
        for rho in (0.0, 2.0):
            for mask, bytes_per in ((0, 48), (1, 96), (7, 432)):
                cls = [rb.prepare(nr, feet, H, 0.01, rho, tw, pos, rot, null, [0, 0, 30., 0, 0, 0],
                                  [1., 10.], mask=mask)[0] for tw in tws]
                ms = timeit(lambda i: cls[i % 2](), iters=20, warm=3)
                row(f"fused rollout rho={rho} out_mask={mask} ({bytes_per} B/eval)", ms, n, bytes_per)
                del cls
                torch.cuda.empty_cache()
        del tws, pos, rot, null
        torch.cuda.empty_cache()
    # --- rollout: warps per 32-chain tile (BLF_CCM_TUNE_ROLLOUT_SPLIT) at configs[2] size ---------
    for nr, feet, H in ((4096, 2, 100), (16384, 2, 100)):
        chains, n = nr * feet, nr * feet * H
        st = syn.make_states(chains, seed=48)
        tile = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).cuda()
        pos, rot, null = tile(st["poses"][:, :3]), tile(st["poses"][:, 3:]), tile(st["null_poses"])
        tws = [rnd(6, n) for _ in range(2)]
        print(f"=== rollout split sweep {nr} x {feet} x {H} ===")
        for split in (1, 2, 4, 8):
            bs = make_batch(BLF_CCM_TUNE_ROLLOUT_SPLIT=split)
            rbs = RolloutBatch(bs)
            for rho in (0.0, 2.0):
                for mask, bytes_per in ((0, 48), (7, 432)):
                    cls = [rbs.prepare(nr, feet, H, 0.01, rho, tw, pos, rot, null, [0, 0, 30., 0, 0, 0],
                                       [1., 10.], mask=mask)[0] for tw in tws]
                    ms = timeit(lambda i: cls[i % 2](), iters=50, warm=5)
                    row(f"split={split} rho={rho} out_mask={mask}", ms, n, bytes_per)
                    del cls
        os.environ.pop("BLF_CCM_TUNE_ROLLOUT_SPLIT", None)
        for ws, label in ((1, "warp-specialised, third form (TMA twists, fused reduction)"), (2, "plain / split (auto)")):
            bs = make_batch(BLF_CCM_TUNE_ROLLOUT_WS=ws)
            rbs = RolloutBatch(bs)
            for rho in (0.0, 0.01, 2.0):
                cls = [rbs.prepare(nr, feet, H, 0.01, rho, tw, pos, rot, null, [0, 0, 30., 0, 0, 0],
                                   [1., 10.], mask=0)[0] for tw in tws]
                ms = timeit(lambda i: cls[i % 2](), iters=50, warm=5)
                row(f"cost-only rho={rho} {label}", ms, n, 48)
                del cls
        os.environ.pop("BLF_CCM_TUNE_ROLLOUT_WS", None)
        del tws, pos, rot, null
        torch.cuda.empty_cache()
    # --- J^T wrench --------------------------------------------------------------------------------
    gf_only()


def gf_only():
    """J^T wrench accumulation: wide Jacobians (lanes own columns) and narrow ones (lane groups own
    whole systems, ccm_genforce_packed_kernel) beside the column-per-lane kernel they replace."""
    from bipedal_locomotion_framework_b200.system import GeneralizedForceBatch
    rnd = lambda *s: torch.rand(s, dtype=torch.float64, device="cuda") * 2 - 1
    for no_pack, stages in ((0, 0), (0, 4), (1, 0)):
        b = make_batch(BLF_CCM_TUNE_NO_PACK=no_pack, BLF_CCM_TUNE_GF_STAGES=stages)
        gf = GeneralizedForceBatch(b)
        shapes = ((409600, 2, 29), (1 << 21, 2, 29), (1 << 20, 4, 38), (1 << 21, 1, 6), (1 << 21, 2, 6),
                  (409600, 2, 6), (1 << 20, 2, 12), (409600, 2, 12), (1 << 20, 2, 16), (1 << 21, 2, 4),
                  (1 << 19, 8, 6), (1 << 20, 4, 12))
        for ns, cps, ncols in shapes:
            if (no_pack or stages) and ncols > 16:
                continue
            n = ns * cps
            st = syn.make_states(min(n, 1 << 18), seed=49)
            reps = (n + st["n"] - 1) // st["n"]
            pl = torch.from_numpy(np.ascontiguousarray(np.tile(
                syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]), (1, reps))[:, :n])).cuda()
            nb = 2 if n * 48 * ncols > (256 << 20) else 3      # rotating sets: never L2-resident
            Js = [rnd(n, 6, ncols) for _ in range(nb)]
            base = rnd(ns, ncols)
            outs = [torch.empty_like(base) for _ in range(nb)]
            cls = [gf.prepare(cps, ncols, pl, Js[j], base, out=outs[j])[0] for j in range(nb)]
            ms = timeit(lambda i: cls[i % nb](), iters=50, warm=5)
            per_contact = 200 + 48 * ncols + 16 * ncols / cps
            row(f"J^T wrench systems={ns} contacts/system={cps} ncols={ncols}"
                f"{' [column-per-lane kernel forced]' if no_pack else ''}{' [four-stage ring]' if stages else ''}",
                ms, n, per_contact)
            del Js, base, outs, cls, pl
            torch.cuda.empty_cache()
    os.environ.pop("BLF_CCM_TUNE_NO_PACK", None)
    os.environ.pop("BLF_CCM_TUNE_GF_STAGES", None)


def dyn_only():
    """Mass-matrix solve (the end of FloatingBaseDynamicalSystem::dynamics) and the whole step.
    Bytes per system: the lower triangle LLT reads (nc(nc+1)/2) + known in + acc out (+ torques);
    the dense matrix the caller hands over is nc*nc -- both fractions are printed."""
    from bipedal_locomotion_framework_b200.system import FloatingBaseDynamicsBatch
    b = make_batch()
    dyn = FloatingBaseDynamicsBatch(b)
    rnd = lambda *s: torch.rand(s, dtype=torch.float64, device="cuda") * 2 - 1
    shapes = ((409600, 29), (1 << 20, 29), (1 << 20, 18), (1 << 21, 12), (1 << 22, 6), (1 << 19, 31),
              (1 << 20, 23), (1 << 20, 24), (1 << 21, 7), (1 << 21, 15), (1 << 18, 38), (1 << 18, 44), (1 << 17, 59), (1 << 17, 64), (1 << 15, 80))
    only = [int(x) if x != "none" else -1 for x in os.environ.get("DYN_NC", "").split(",") if x]
    euler_only = os.environ.get("DYN_EULER_ONLY") == "1"
    for ns, nc in shapes:
        if only and nc not in only:
            continue
        nb = 3
        Ms = []
        for _ in range(nb):
            A = rnd(ns, nc, nc)
            M = torch.bmm(A, A.transpose(1, 2)) / nc
            del A
            M.diagonal(dim1=1, dim2=2).add_(0.5)
            Ms.append(M)
        known = rnd(ns, nc)
        tau = rnd(ns, nc - 6) if nc > 6 else None
        outs = [torch.empty_like(known) for _ in range(nb)]
        cls = [dyn.prepare_solve(Ms[j], known, tau, out=outs[j])[0] for j in range(nb)]
        ms = timeit(lambda i: cls[i % nb](), iters=30, warm=5)
        tri = 8 * (nc * (nc + 1) // 2 + 2 * nc + max(nc - 6, 0))
        dense = 8 * (nc * nc + 2 * nc + max(nc - 6, 0))
        gbs_t, gbs_d = ns * tri / (ms * 1e-3) / 1e9, ns * dense / (ms * 1e-3) / 1e9
        flops = ns * (nc ** 3 / 3 + 2 * nc * nc) / (ms * 1e-3) / 1e12
        print(f"mass-matrix solve systems={ns:8d} nc={nc:3d}  {ms*1e3:9.1f} us  {ns/ms/1e3:8.1f} M systems/s  "
              f"lower-triangle {gbs_t:7.1f} GB/s {gbs_t/PEAK*100:5.1f} %   dense {gbs_d:7.1f} GB/s {gbs_d/PEAK*100:5.1f} %   "
              f"{flops:5.2f} TFLOP/s", flush=True)
        del Ms, outs, cls
        torch.cuda.empty_cache()
    # the whole step at the MPC batch size: 409600 systems x 2 contacts, 6 + 23 DoF
    for ns, cps, nc in ((409600, 2, 29), (409600, 2, 12), (1 << 21, 2, 29), (1 << 22, 1, 6)):
        n = ns * cps
        st = syn.make_states(min(n, 1 << 18), seed=49)
        reps = (n + st["n"] - 1) // st["n"]
        pl = torch.from_numpy(np.ascontiguousarray(np.tile(
            syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]), (1, reps))[:, :n])).cuda()
        nb = 3
        Js = [rnd(n, 6, nc) for _ in range(nb)]
        Ms = []
        for _ in range(nb):
            A = rnd(ns, nc, nc)
            M = torch.bmm(A, A.transpose(1, 2)) / nc
            del A
            M.diagonal(dim1=1, dim2=2).add_(0.5)
            Ms.append(M)
        bias, tau = rnd(ns, nc), (rnd(ns, nc - 6) if nc > 6 else None)
        outs = [torch.empty_like(bias) for _ in range(nb)]
        cls = [dyn.prepare_acceleration(cps, pl, Js[j], bias, Ms[j], tau, out=outs[j])[0] for j in range(nb)]
        ms = timeit(lambda i: cls[i % nb](), iters=(3 if euler_only else 30), warm=(1 if euler_only else 5))
        per_sys = cps * (200 + 48 * nc) + 8 * (nc * (nc + 1) // 2 + 2 * nc + (nc - 6))
        gbs = ns * per_sys / (ms * 1e-3) / 1e9
        if not euler_only:
            print(f"floating-base acceleration systems={ns} contacts/system={cps} nc={nc}  {ms*1e3:9.1f} us  "
              f"{ns/ms/1e3:8.1f} M systems/s  {gbs:7.1f} GB/s {gbs/PEAK*100:5.1f} % (lower-triangle bytes)", flush=True)
        # one ForwardEuler step of the whole floating-base state: (5 nc + 12) doubles per system
        nu, jp, bp = rnd(ns, nc), (rnd(ns, nc - 6) if nc > 6 else None), rnd(ns, 3)
        br = torch.eye(3, dtype=torch.float64, device="cuda").reshape(1, 9).repeat(ns, 1)
        for rho in (0.01, 0.0):
            ec = dyn.prepare_euler_step(rho, 1e-5, outs[0], nu, jp, bp, br)
            ems = timeit(lambda i: ec(), iters=30, warm=5)
            eb = 8 * (5 * nc + 12)
            print(f"floating-base Euler step systems={ns} nc={nc} rho={rho}  {ems*1e3:9.1f} us  {ns/ems/1e3:8.1f} M systems/s  "
                  f"{ns*eb/(ems*1e-3)/1e9:7.1f} GB/s {ns*eb/(ems*1e-3)/1e9/PEAK*100:5.1f} %", flush=True)
        del Js, Ms, outs, cls, pl
        torch.cuda.empty_cache()


def main():
    if "--rls-only" in sys.argv:
        return rls_only()
    if "--dyn-only" in sys.argv:
        return dyn_only()
    if "--sys-only" in sys.argv:
        return sys_only()
    if "--gf-only" in sys.argv:
        return gf_only()
    sizes = {"cfg3 819200": 2 * 4096 * 100, "8M": 1 << 23}
    NS = 3
    for label, n in sizes.items():
        st = syn.make_states(min(n, 1 << 20), seed=45)
        reps = (n + st["n"] - 1) // st["n"]
        pl = np.tile(syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"]), (1, reps))[:, :n]
        planes = [torch.from_numpy(np.ascontiguousarray(pl)).cuda() for _ in range(NS)]
        het = syn.make_states(min(n, 1 << 20), seed=46, heterogeneous=True)
        prm = torch.from_numpy(np.ascontiguousarray(np.tile(het["params"].T, (1, reps))[:, :n])).cuda()
        aos = [torch.from_numpy(np.ascontiguousarray(np.tile(st[k], (reps, 1))[:n])).cuda()
               for k in ("twists", "poses", "null_poses")]
        prm_aos = prm.T.contiguous()
        print(f"\n=== n = {n} ({label}); peak {PEAK} GB/s ===")
        b = make_batch()
        outs = [b.alloc_soa_outputs(n, FULL) for _ in range(NS)]
        cl = [b.prepare_soa(planes[j], None, FULL, out=outs[j])[0] for j in range(NS)]
        ms = timeit(lambda i: cl[i % NS]())
        row("soa full uniform", ms, n, 600)
        cl = [b.prepare_soa(planes[j], prm, FULL, out=outs[j])[0] for j in range(NS)]
        ms = timeit(lambda i: cl[i % NS]())
        row("soa full heterogeneous", ms, n, 632)
        rl = 200 if n % 200 == 0 else 256
        cl = [b.prepare_rollout(planes[j], rl, [0, 0, 30., 0, 0, 0], [1., 10.], mask=FULL, out=outs[j],
                                want_cost=False)[0] for j in range(NS)]
        ms = timeit(lambda i: cl[i % NS]())
        row(f"rollout({rl}) full + cost + argmin (2 launches)", ms, n, 600)
        cl = [b.prepare_rollout(planes[j], rl, [0, 0, 30., 0, 0, 0], [1., 10.], mask=0)[0] for j in range(NS)]
        ms = timeit(lambda i: cl[i % NS]())
        row(f"rollout({rl}) cost only (25 planes in)", ms, n, 200)
        del outs
        outs = [b.alloc_soa_outputs(n, WRENCH) for _ in range(NS)]
        cl = [b.prepare_soa(planes[j], None, WRENCH, out=outs[j])[0] for j in range(NS)]
        ms = timeit(lambda i: cl[i % NS]())
        row("soa wrench-only uniform", ms, n, 248)
        del outs
        outs = [b.alloc_aos_outputs(n, FULL) for _ in range(2)]
        ms = timeit(lambda i: b.evaluate_aos(aos[0], aos[1], aos[2], None, FULL, out=outs[i % 2]))
        row("aos full uniform (624 B touched)", ms, n, 600)
        ms = timeit(lambda i: b.evaluate_aos(aos[0], aos[1], aos[2], prm_aos, FULL, out=outs[i % 2]))
        row("aos full heterogeneous", ms, n, 632)
        del outs
        outs = [b.alloc_aos_outputs(n, WRENCH) for _ in range(2)]
        ms = timeit(lambda i: b.evaluate_aos(aos[0], aos[1], aos[2], None, WRENCH, out=outs[i % 2]))
        row("aos wrench-only", ms, n, 248)
        # recursive least squares (section 8f row 1)
        from bipedal_locomotion_framework_b200.estimators import RecursiveLeastSquareBatch
        rls = RecursiveLeastSquareBatch(b, [1.0, 1.0, 1.0, 0.01, 0.01, 0.01], 0.99)
        th = torch.rand((2, n), dtype=torch.float64, device="cuda") * 1e3 + 10
        P = torch.zeros((4, n), dtype=torch.float64, device="cuda"); P[0] = 1e6; P[3] = 1e4
        zz = torch.randn((6, n), dtype=torch.float64, device="cuda")
        Yp = torch.randn((12, n), dtype=torch.float64, device="cuda") * 1e-2
        rsets = [(Yp.clone(), zz.clone(), th.clone(), P.clone()) for _ in range(2 if n < (1 << 22) else 1)]
        rcalls = [rls.prepare_advance(*s_) for s_ in rsets]
        ms = timeit(lambda i: rcalls[i % len(rcalls)](), iters=100)
        row("rls advance p=2 m=6 (regressor planes in)", ms, n, 240)
        for s_ in rsets:
            s_[3].zero_(); s_[3][0] = 1e6; s_[3][3] = 1e4
        rcalls = [rls.prepare_advance_contacts(planes[k % NS], s_[1], s_[2], s_[3])
                  for k, s_ in enumerate(rsets)]
        ms = timeit(lambda i: rcalls[i % len(rcalls)](), iters=100)
        row("rls fused contact identification (state planes in)", ms, n, 344)
        del th, P, zz, Yp, rsets, rcalls
        del outs, planes, aos, prm, prm_aos
        torch.cuda.empty_cache()

    # torch copy reference point (same method as MEASURED_PEAKS)
    x = torch.empty(1 << 28, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)
    ms = timeit(lambda i: y.copy_(x), iters=10, warm=3)
    print(f"\ntorch copy 2 GiB+2 GiB: {2 * x.numel() * 8 / (ms * 1e-3) / 1e9:.1f} GB/s")
    del x, y

    # host pipeline chunk sweep (config 3, pinned)
    n = 2 * 4096 * 100
    st = syn.make_states(n, seed=45)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h = [pin(st[k]) for k in ("twists", "poses", "null_poses")]
    ho = {"wrench": torch.empty((n, 6), dtype=torch.float64).pin_memory(),
          "autodyn": torch.empty((n, 6), dtype=torch.float64).pin_memory(),
          "ctrl": torch.empty((n, 36), dtype=torch.float64).pin_memory(), "regressor": None}
    b = make_batch()
    print("\nhost pipeline (pinned, 240 B in + 384 B out per eval):")
    for chunk in (8192, 16384, 32768, 65536, 131072, 819200):
        b.set_host_chunk(chunk)
        for _ in range(2):
            b.evaluate_host(h[0], h[1], h[2], None, FULL, out=ho)
        t0 = time.perf_counter()
        for _ in range(5):
            b.evaluate_host(h[0], h[1], h[2], None, FULL, out=ho)
        dt = (time.perf_counter() - t0) / 5
        print(f"  chunk {chunk:7d}: {dt*1e3:7.2f} ms  {n/dt/1e6:7.1f} M evals/s  "
              f"h2d {n*240/dt/1e9:5.1f} GB/s  d2h {n*384/dt/1e9:5.1f} GB/s", flush=True)


if __name__ == "__main__":
    main()
