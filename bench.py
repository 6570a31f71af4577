#!/usr/bin/env python
"""bench.py -- contact evals/sec (wrench + 6x6 Jacobians, FP64) of the batched
ContinuousContactModel evaluation at 1/2/4/8 B200, with roofline, CPU baseline and end-to-end numbers.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one batch of synthetic contact states.

Headline (`value`, every N): BASELINE.json configs[4] -- STRONG scaling over 2^28 contact states,
wrench + autonomous dynamics + dense 6x6 control matrix, uniform foot, SoA planes (600 algorithmic
bytes per evaluation).  The batch is 2^20 rollouts of 256 evaluations (2 feet x 128 steps),
block-partitioned by rollout over the N ranks; every timed step is ONE call of
blf_ccm_rollout_cost_argmin_soa per rank: evaluate the shard, reduce the per-rollout cost in the
kernel's epilogue, arg-min, and -- for N > 1 -- exchange the 16-byte (cost, index) pair with every
peer over NVLink peer memory INSIDE the last block of the reduction kernel.  The collective is
therefore inside the timed value; every timed step's global arg-min is checked afterwards against
an NCCL all-gather of the same per-rank pairs (`exchange_check`).

Extra records on the same line (never part of `value`): configs[3] (64 M heterogeneous states +
arg-min, strong), configs[2] (sampling-MPC batch 2 x 4096 x 100 per GPU, weak: plain evaluation,
MPC step, fused integrate->contact->cost rollout), the rows next to the path, `e2e` through
blf_ccm_eval_batch_host with HOST buffers, `cpu_baseline`, `sustained` (>= 1 s back to back).

Prints ONE JSON line on rank 0.  --dump-outputs DIR also writes what the headline's last timed step
handed its caller as .npy files (dump_outputs), so that two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FEET, SAMPLES, HORIZON = 2, 4096, 100
N_MPC = FEET * SAMPLES * HORIZON              # 819 200: configs[2] per GPU
MPC_ROLLOUT_LEN = FEET * HORIZON              # 200
HEAD_ROLLOUTS, HEAD_ROLLOUT_LEN = 1 << 20, 256   # configs[4]: 2^20 rollouts x (2 feet x 128 steps) = 2^28
HET_ROLLOUTS, HET_ROLLOUT_LEN = 335544, 200      # configs[3]: 67 108 800 ~ 2^26 heterogeneous states
CPU_SAMPLE = N_MPC                            # states per CPU-arm step (bounded sample of the workload)
E2E_PER_RANK = 1 << 21                        # host-buffer leg: states per rank and step
BYTES_FULL_UNIFORM, BYTES_FULL_HET = 600, 632  # BASELINE.md section 3
METRIC = "contact evals/sec (wrench+6x6 Jacobians, FP64)"
UNIT = "evals/s"
REF_WRENCH, WEIGHTS = [0.0, 0.0, 30.0, 0.0, 0.0, 0.0], [1.0, 10.0]
DUMP_STATES = 1 << 16                         # --dump-outputs: states of the fixed, seeded output sample

_JSON_OUT = None


def emit(line: dict) -> None:
    """The one JSON line, on the process's original stdout."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def shared_config(world: int) -> dict:
    """`config` of BOTH arms (ours and --impl reference): what is measured, nothing arm-specific."""
    return {
        "workload": ("configs[4]: strong scaling, 2^28 contact states, wrench + autonomous dynamics + "
                     "6x6 control matrix, uniform foot geometry and stiffness/damping; 2^20 rollouts "
                     "x 256 evaluations, per-rollout cost + arg-min"),
        "evals_per_step": HEAD_ROLLOUTS * HEAD_ROLLOUT_LEN,
        "rollouts": HEAD_ROLLOUTS, "rollout_len": HEAD_ROLLOUT_LEN,
        "parallelism": f"rollout-sharded x{world}",
        "seed": 46,
    }


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _traffic(kernel: str):
    """dram bytes per evaluation of the named kernel from the committed ncu --set full capture
    (profiles/roofline_traffic.json; regenerated whenever that kernel changes), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            d = json.load(f)
        return d.get("dram_bytes_per_eval", {}).get(kernel)
    except Exception:
        return None


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the bench runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting",
               0x100: "display_clock_setting", 0x10: "sync_boost"}

    def __init__(self, index: int, period: float = 0.003):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples = []
        self.stop_flag = False
        self.ok = False
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), clk, rs))
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self, t0: float, t1: float) -> dict:
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        window = "timed"
        if len(inside) < 3:
            inside = [s for s in self.samples if s[0] <= t1][-8:] or list(self.samples)
            window = "warmup+timed (timed region shorter than 3 samples)"
        clks = sorted(s[1] for s in inside) or [0]
        bits = 0
        for s in inside:
            bits |= s[2]
        reasons = [name for bit, name in self.REASONS.items() if bits & bit]
        return {"sm_mhz": clks[len(clks) // 2], "sm_min_mhz": clks[0], "sm_max_mhz": self.sm_max,
                "reasons": reasons, "samples": len(inside), "window": window}


# --------------------------------------------------------------------------------------------------
# CPU arm (oracle): bench.py may execute oracle/ only here and in the parity checks
# --------------------------------------------------------------------------------------------------

def _cpu_impl(prefer_reference: bool = True):
    """(module, kind, what): oracle/_ref (the reference's own sources compiled against stand-in
    Eigen/iDynTree headers, kind "reference") when it was built, else the C port (kind "port")."""
    from oracle import ccm_oracle, ref_binding
    if prefer_reference and ref_binding.usable():
        return ref_binding, "reference", ("oracle/_ref: the reference's ContinuousContactModel.cpp compiled in place "
                                          "against stand-in Eigen/iDynTree headers (eager evaluation), g++ -O3 -DNDEBUG = CMake Release")
    ccm_oracle.build()
    return ccm_oracle, "port", "oracle/ccm_oracle.c per-instance path, gcc -O2 -ffp-contract=off"


def cpu_reference_pass(st, nthreads: int, min_seconds: float, mask: int = 7, prefer_reference: bool = True):
    """Time the reference's per-instance path (threaded) on the given states."""
    impl, kind, what = _cpu_impl(prefer_reference)
    n = st["twists"].shape[0]
    best = None
    spent = 0.0
    passes = 0
    while spent < min_seconds or passes < 2:
        t0 = time.perf_counter()
        impl.eval_batch_states(st, mask=mask, nthreads=nthreads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        spent += dt
        passes += 1
    return n / best, passes, spent, kind, what


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from bipedal_locomotion_framework_b200 import synthetic as syn
    cores = os.cpu_count() or 1
    sample_n = CPU_SAMPLE
    st = syn.make_states(sample_n, seed=46)
    impl, kind, what = _cpu_impl()
    for _ in range(max(1, min(args.warmup, 3))):
        impl.eval_batch_states(st, mask=7, nthreads=cores)
    steps = max(1, args.steps)  # each step is one 819 200-state pass
    t0 = time.perf_counter()
    for _ in range(steps):
        impl.eval_batch_states(st, mask=7, nthreads=cores)
    dt = time.perf_counter() - t0
    value = sample_n * steps / dt
    sample = (f"{steps} passes over a {sample_n}-state sample of the workload (same state distribution), "
              f"{cores} threads, one model object per thread: setState, setNullForceTransform, "
              f"getContactWrench, getAutonomousDynamics, getControlMatrix per state; {what}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": dt / steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": shared_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": ("the reference's own sources, compiled from BLF_REFERENCE_ROOT into oracle/_ref against stand-in "
                 "Eigen/iDynTree headers (the real libraries are absent from the image); a CPU rate does not "
                 "depend on the batch size, so each step times a bounded sample of the 2^28-state workload"
                 if kind == "reference"
                 else "oracle/_ref was not built (no BLF_REFERENCE_ROOT at build time): C port timed"),
    }
    if kind == "reference":  # the leaner C restatement beside it, for scale
        v, passes, spent, _, pwhat = cpu_reference_pass(st, cores, 2.0, prefer_reference=False)
        line["cpu_baseline"]["port_value"] = v
        line["cpu_baseline"]["port_sample"] = f"best of {passes} passes, {pwhat}"
    emit(line)
    return 0


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------

class Ctx:
    """Process-wide state of one bench rank."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        from bipedal_locomotion_framework_b200 import sharding
        from bipedal_locomotion_framework_b200 import synthetic as syn
        from bipedal_locomotion_framework_b200.contact_models import ContinuousContactModelBatch

        self.torch, self.dist, self.sharding, self.syn = torch, dist, sharding, syn
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the contact-model backend has no CPU path")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        if args.gpus != self.world and self.rank == 0:
            print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={self.world}; using {self.world}", file=sys.stderr)
        self.batch = ContinuousContactModelBatch(self.local)
        self.batch.set_uniform_params(*syn.REFERENCE_TEST_PARAMS)
        self.peak, self.peak_src = _peaks()
        self.args = args
        # the only exchange of the path: every rank's 16-byte (cost, index) pair, through the peers'
        # mailboxes over NVLink (fused into the reduction kernel); NCCL all-gather as the fallback
        self.peer, self.peer_note = None, None
        if self.world > 1 and not args.nccl_argmin:
            try:
                self.peer = sharding.PeerArgmin(self.batch, self.world, self.rank, dist)
            except Exception as e:   # e.g. CUDA IPC not permitted in this container
                self.peer_note = f"peer-memory mailbox unavailable ({e}); NCCL all-gather used"
        if self.world > 1:   # the choice must be the same on every rank
            flag = torch.tensor([1 if self.peer is not None else 0], device=self.dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                self.peer = None
        self.sampler = ClockSampler(self.local)
        self.sampler.start()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def min_flag(self, ok: bool) -> bool:
        if self.world == 1:
            return bool(ok)
        t = self.torch.tensor([1 if ok else 0], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t.item()))

    def collective_name(self):
        if self.world == 1:
            return "none (1 GPU)"
        if self.peer is not None:
            return ("peer-memory mailbox over NVLink, fused into the last block of the cost-reduction kernel "
                    "(blf_ccm_rollout_set_exchange): no extra launch, no collective library")
        return "nccl all_gather 16 B/rank + device arg-min"

    def close(self):
        self.sampler.stop_flag = True
        if self.world > 1:
            self.dist.destroy_process_group()


def rollout_workload(cx: Ctx, what: str, total_rollouts: int, rollout_len: int, het: bool, K: int, W: int,
                     seed: int, sustain_s: float = 0.0, nsets: int = 1, host_planes=None,
                     force_windows: int = 0, dump_dir: str | None = None) -> dict:
    """One sharded sampling-MPC evaluation workload, timed as the contract says.

    Rank r owns rollouts [first, first+count) of `total_rollouts`.  A step = one
    blf_ccm_rollout_cost_argmin_soa call on the shard (full outputs + per-rollout cost + arg-min)
    with the peer exchange fused into its reduction kernel.  The reference force changes a little
    every step, so every step has its own costs and the exchange of one step cannot be mistaken
    for another's; local and global pairs of every step land in their own slots and are compared
    with an NCCL all-gather arg-min afterwards (outside the timed region)."""
    import ctypes as C

    from bipedal_locomotion_framework_b200 import _capi
    from bipedal_locomotion_framework_b200.contact_models import FULL, ContinuousContactModelBatch
    torch, dist, syn, batch = cx.torch, cx.dist, cx.syn, cx.batch
    world, rank, dev = cx.world, cx.rank, cx.dev
    first, count = cx.sharding.shard_rollouts(total_rollouts, world, rank)
    n = count * rollout_len
    bytes_per = BYTES_FULL_HET if het else BYTES_FULL_UNIFORM

    # ---- memory: the whole shard resident (inputs + outputs); if the outputs do not fit, a window
    # of the outputs is reused by several sub-calls per step (stated in the result)
    in_planes = 27 + (4 if het else 0)
    free_b = torch.cuda.mem_get_info(dev)[0]
    need_in = n * in_planes * 8 * nsets
    windows = max(1, force_windows)
    while windows < 64 and need_in + (n // windows + rollout_len) * 48 * 8 * nsets + (6 << 30) > free_b:
        windows *= 2
    roll_win = (count + windows - 1) // windows
    n_win = roll_win * rollout_len

    sets = []
    for j in range(nsets):
        if host_planes is not None:     # configs[2]: the seeded numpy stream, same bits as the CPU arm
            pl, prm = torch.from_numpy(host_planes).to(dev), None
            pl = [pl[i] for i in range(30)]
        else:
            pl, prm = syn.make_planes_torch(n, dev, seed=seed + 1000 * rank + 7 * j, heterogeneous=het)
        out = batch.alloc_soa_outputs(min(n, n_win), FULL)
        cost = torch.empty(count, dtype=torch.float64, device=dev)
        sets.append((pl, prm, out, cost))
    torch.cuda.synchronize()

    T = W + K + 8                                           # slots: warm-up, timed, blocked-peer probe
    hist_l = torch.zeros((T, 2), dtype=torch.int64, device=dev)   # this rank's pair of every step
    hist_g = torch.zeros((T, 2), dtype=torch.int64, device=dev)   # global pair of every step
    sub_best = torch.zeros((windows, 2), dtype=torch.int64, device=dev)
    ref = np.ascontiguousarray(REF_WRENCH, dtype=np.float64)
    wts = np.ascontiguousarray(WEIGHTS, dtype=np.float64)
    lib = _capi.lib()
    fn = lib.blf_ccm_rollout_cost_argmin_soa
    pp = ContinuousContactModelBatch._plane_ptrs
    stream = batch._stream()
    hp = batch.handle.ptr
    fused = cx.peer is not None and windows == 1
    hl0, hg0 = hist_l.data_ptr(), hist_g.data_ptr()   # slot i of either history = base + 16 i
    state = {"last": 0}

    def view(pl, a, b):
        return [None if p is None else p[a:b] for p in pl]

    bound = []   # per set, per window: argument list with the `best` pointer left open (index 13)
    for pl, prm, out, cost in sets:
        per = []
        for w in range(windows):
            r0 = w * roll_win
            r1 = min(count, r0 + roll_win)
            if r1 <= r0:
                continue
            a, b = r0 * rollout_len, r1 * rollout_len
            o = {k: (None if v is None else (v[: b - a] if k == "ctrl" else v[:, : b - a])) for k, v in out.items()}
            keep = (view(pl, a, b), None if prm is None else view(prm, a, b), o)
            per.append(([hp, r1 - r0, rollout_len, pp(keep[0], 30), pp(keep[1], 4), FULL,
                         pp(o["wrench"], 6), pp(o["autodyn"], 6), o["ctrl"].data_ptr(),
                         ref.ctypes.data_as(C.c_void_p), wts.ctypes.data_as(C.c_void_p), first + r0,
                         cost[r0:r1].data_ptr(), None, stream], keep))
        bound.append(per)

    def step(i: int, delay: float = 0.0):
        """step i (slot i of the history buffers)"""
        ref[2] = 30.0 + 1e-3 * (i % 97)
        per = bound[i % nsets]
        state["last"] = i
        if delay:
            time.sleep(delay)
        if fused:
            rc = lib.blf_ccm_rollout_set_exchange(hp, hg0 + 16 * i)
            if rc:
                _capi.check(rc)
        if len(per) == 1:
            a = per[0][0]
            a[13] = hl0 + 16 * i
            rc = fn(*a)
            if rc:
                _capi.check(rc)
        else:
            for w, (a, _) in enumerate(per):
                a[13] = sub_best[w].data_ptr()
                rc = fn(*a)
                if rc:
                    _capi.check(rc)
            _capi.check(lib.blf_ccm_argmin_pairs(hp, len(per), sub_best.data_ptr(), hist_l[i].data_ptr(), stream))
        if world > 1 and not fused:
            if cx.peer is not None:
                cx.peer.exchange(hist_l[i], out=hist_g[i])
            else:
                g = cx.sharding.all_gather_pairs(hist_l[i], world, dist)
                _capi.check(lib.blf_ccm_argmin_pairs(hp, world, g.data_ptr(), hist_g[i].data_ptr(), stream))

    for i in range(W):
        step(i)
    cx.barrier()
    l0 = batch.handle.launch_count
    t_host0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(W, W + K):
        step(i)
    e1.record()
    cx.barrier()
    t_host1 = time.perf_counter()
    launches = batch.handle.launch_count - l0
    my_ms = e0.elapsed_time(e1)
    ms = cx.max_over_ranks(my_ms)
    clocks = cx.sampler.summary(t_host0, t_host1)
    if dump_dir is not None and rank == 0:
        last = W + K - 1
        dump_outputs(dump_dir, torch, batch, bound[last % nsets][-1][1][2], sets[last % nsets][3],
                     hist_g[last] if world > 1 else hist_l[last])

    # ---- blocked-peer probe: the last rank arrives 50 ms late, four times; nobody may mix epochs
    probe_steps = 4 if world > 1 else 0
    for j in range(probe_steps):
        step(W + K + j, delay=0.05 if rank == world - 1 else 0.0)
    cx.barrier()
    if fused:
        _capi.check(lib.blf_ccm_rollout_set_exchange(hp, None))

    # ---- every step's global pair against an NCCL all-gather of the same local pairs -------------
    exchange_check = None
    if world > 1:
        used = W + K + probe_steps
        g = torch.empty((world, T, 2), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(g.view(-1), hist_l.view(-1))
        gl = g.cpu().numpy()[:, :used]
        costs = gl[..., 0].copy().view(np.float64)
        idx = gl[..., 1]
        costs = np.where(idx >= 0, costs, np.inf)
        want_c = costs.min(axis=0)
        want_i = np.where(costs == want_c[None, :], idx, np.iinfo(np.int64).max).min(axis=0)
        got = hist_g.cpu().numpy()[:used]
        got_c, got_i = got[:, 0].copy().view(np.float64), got[:, 1]
        ok_all = bool(np.array_equal(got_c, want_c) and np.array_equal(got_i, want_i))
        timed = slice(W, W + K)
        ok_timed = bool(np.array_equal(got_c[timed], want_c[timed]) and np.array_equal(got_i[timed], want_i[timed]))
        pr = slice(W + K, used)
        ok_probe = bool(np.array_equal(got_c[pr], want_c[pr]) and np.array_equal(got_i[pr], want_i[pr]))
        exchange_check = {
            "steps": K, "ok": cx.min_flag(ok_timed),
            "how": "global pair of every timed step == arg-min (lowest-index tie-break) of an NCCL all-gather of "
                   "the per-rank pairs of that step, bit for bit, on every rank",
            "distinct_costs": int(len(np.unique(want_c[timed]))),
            "blocked_peer_probe": {"delay_ms": 50, "steps": probe_steps, "late_rank": world - 1,
                                   "ok": cx.min_flag(ok_probe)},
            "all_ok": cx.min_flag(ok_all), "collective": cx.collective_name()}

    # ---- parity on the same device bits: sampled states + whole sampled rollouts (cost) ----------
    from oracle import ccm_oracle
    torch.cuda.synchronize()
    pl, prm, out, cost = sets[state["last"] % nsets]   # the set (and `ref`) of the last executed step
    # (the last window's outputs are what `out` holds: sample inside it)
    lastw = bound[state["last"] % nsets][-1][1]
    wpl, wprm, wout = lastw
    nw = wout["ctrl"].shape[0]
    stride = 1 if nw <= (1 << 16) else max(1, (nw // (1 << 15)) | 1)
    idx = torch.arange(0, nw, stride, device=dev)
    stt = syn.sample_states_from_planes(wpl, wprm, idx)
    cores = os.cpu_count() or 1
    refo = ccm_oracle.eval_batch_states(stt, mask=7, nthreads=cores)
    got = {"wrench": torch.stack([p[idx] for p in wout["wrench"]], 1).cpu().numpy(),
           "autodyn": torch.stack([p[idx] for p in wout["autodyn"]], 1).cpu().numpy(),
           "ctrl": wout["ctrl"][idx].cpu().numpy()}
    worst = 0.0
    for key, blocks in (("wrench", [slice(0, 3), slice(3, 6)]), ("autodyn", [slice(0, 3), slice(3, 6)]),
                        ("ctrl", [slice(6 * q + 3 * (q // 3), 6 * q + 3 * (q // 3) + 3) for q in range(6)])):
        for sl in blocks:
            num = np.abs(got[key][:, sl] - refo[key][:, sl]).max(axis=1)
            den = np.maximum(np.abs(refo[key][:, sl]).max(axis=1), 1e-300)
            worst = max(worst, float(np.where(num == 0, 0, num / den).max()))
    zmask = np.ones(36, dtype=bool)
    for q in range(3):
        zmask[6 * q + q] = False
        zmask[6 * (3 + q) + 3: 6 * (3 + q) + 6] = False
    zeros_ok = bool((got["ctrl"][:, zmask].view(np.int64) == 0).all())   # exactly +0.0
    # cost of 16 whole rollouts of the last step
    rsel = np.unique(np.linspace(0, count - 1, 16).astype(np.int64)) if count > 0 else np.zeros(0, np.int64)
    cost_err = 0.0
    if len(rsel):
        ridx = torch.from_numpy((rsel[:, None] * rollout_len + np.arange(rollout_len)[None, :]).reshape(-1)).to(dev)
        sr = syn.sample_states_from_planes(pl, prm, ridx)
        wr = ccm_oracle.eval_batch_states(sr, mask=1, nthreads=cores)["wrench"]
        want = ccm_oracle.rollout_cost(wr, rollout_len, ref, wts)
        gotc = cost.cpu().numpy()[rsel]
        cost_err = float(np.max(np.abs(gotc - want) / np.maximum(np.abs(want), 1e-300)))
    worst_all = cx.max_over_ranks(max(worst, cost_err))
    parity = {"sampled_states_per_rank": int(idx.numel()), "sampled_rollout_costs_per_rank": int(len(rsel)),
              "worst_block_rel_err": cx.max_over_ranks(worst), "worst_cost_rel_err": cx.max_over_ranks(cost_err),
              "structural_zeros_exact": cx.min_flag(zeros_ok), "tol": 1e-12,
              "ok": bool(worst_all <= 1e-12) and cx.min_flag(zeros_ok), "ranks_checked": world,
              "checker": "oracle/ccm_oracle.c on the same device bits"}

    best_pair = hist_g[W + K - 1] if world > 1 else hist_l[W + K - 1]
    bc, bi = batch.decode_best(best_pair)

    # ---- sustained: the same step back to back for >= sustain_s seconds, own clock window --------
    sustained = None
    if sustain_s > 0:
        if fused:
            _capi.check(lib.blf_ccm_rollout_set_exchange(hp, hist_g[0].data_ptr()))
        reps = max(K, int(sustain_s * 1e3 / max(ms / K, 1e-3)) + 1)
        if world > 1:   # the same count on every rank (the exchange is a collective)
            t = torch.tensor([reps], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            reps = int(t.item())
        cx.barrier()
        ts0 = time.perf_counter()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(reps):
            step(W + (i % K))
        s1.record()
        cx.barrier()
        ts1 = time.perf_counter()
        sms = cx.max_over_ranks(s0.elapsed_time(s1))
        sc = cx.sampler.summary(ts0, ts1)
        sustained = {"seconds": sms * 1e-3, "steps": reps, "ms_per_step": sms / reps,
                     "value": total_rollouts * rollout_len * reps / (sms * 1e-3), "unit": UNIT,
                     "frac": bytes_per * n / (sms / reps * 1e-3) / 1e9 / cx.peak, "clocks": sc}
        if fused:
            _capi.check(lib.blf_ccm_rollout_set_exchange(hp, None))

    total = total_rollouts * rollout_len
    gbs = bytes_per * n / (ms / K * 1e-3) / 1e9 if n else 0.0
    res = {"what": what, "value": total * K / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / K, "steps": K,
           "warmup": W, "evals_per_step": total, "evals_per_step_per_gpu": n, "rollouts": total_rollouts,
           "rollout_len": rollout_len, "heterogeneous": het, "gpu_launches": int(launches),
           "output_windows": windows,
           "roofline": {"bound": "hbm", "achieved": gbs, "peak": cx.peak, "unit": "GB/s", "frac": gbs / cx.peak,
                        "algorithmic_bytes_per_eval": bytes_per, "algorithmic_bytes_per_launch": bytes_per * n,
                        "avg_launch_ms": my_ms / K,
                        "note": "rank 0's shard; duration = whole step (evaluation kernel + reduction/exchange "
                                "launch), so the fraction is a lower bound for the evaluation kernel",
                        "peak_source": cx.peak_src},
           "clocks": clocks, "parity": parity, "exchange_check": exchange_check, "collective": cx.collective_name(),
           "argmin": {"cost": bc, "rollout": bi}, "sustained": sustained}
    return res


def dump_outputs(out_dir: str, torch, batch, out: dict, cost, best_pair) -> None:
    """What one step of blf_ccm_rollout_cost_argmin_soa handed its caller, as float64 .npy files: the
    wrench, autonomous dynamics and control matrix of a fixed, seeded sample of the states (indices in
    state_index; within the last output window when the outputs are windowed), every rollout's cost and
    the arg-min pair (best = [cost, rollout]).  About 34 MB for the headline on one GPU."""
    torch.cuda.synchronize()
    n = out["ctrl"].shape[0]
    idx_np = np.unique(np.random.default_rng(2024).integers(0, n, DUMP_STATES))
    idx = torch.from_numpy(idx_np).to(out["ctrl"].device)
    bc, bi = batch.decode_best(best_pair)
    arrays = {"state_index": idx_np, "wrench": out["wrench"][:, idx].T, "autodyn": out["autodyn"][:, idx].T,
              "ctrl": out["ctrl"][idx], "cost": cost, "best": np.array([bc, bi])}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else a
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def eval_only_leg(cx: Ctx, planes_np, K: int, W: int) -> dict:
    """configs[2] per GPU, plain blf_ccm_eval_batch_soa (no epilogue): the kernel of the round-1
    headline, 3 rotating buffer sets so no step finds its 491.5 MB in the 126 MB L2."""
    from bipedal_locomotion_framework_b200.contact_models import FULL
    torch, batch, dev = cx.torch, cx.batch, cx.dev
    n = planes_np.shape[1]
    NSETS = 3
    planes = [torch.from_numpy(planes_np).to(dev) for _ in range(NSETS)]
    outs = [batch.alloc_soa_outputs(n, FULL) for _ in range(NSETS)]
    calls = [batch.prepare_soa(planes[j], None, FULL, out=outs[j])[0] for j in range(NSETS)]
    for i in range(W):
        calls[i % NSETS]()
    cx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        calls[i % NSETS]()
    e1.record()
    cx.barrier()
    my_ms = e0.elapsed_time(e1)
    ms = cx.max_over_ranks(my_ms)
    gbs = BYTES_FULL_UNIFORM * n / (my_ms / K * 1e-3) / 1e9
    return {"what": "configs[2] per GPU (weak): 819 200 states, blf_ccm_eval_batch_soa wrench+autodyn+ctrl, no epilogue",
            "value": cx.world * n * K / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / K, "steps": K,
            "scaling": "weak", "hbm_frac_of_measured": gbs / cx.peak,
            "kernel": "ccm_soa_kernel<WRENCH|AUTODYN|CTRL, uniform, no cost>",
            "traffic_bytes_per_eval_ncu": _traffic("ccm_soa_kernel<7,0,0>")}


def fused_rollout_leg(cx: Ctx, planes_np, K: int, W: int, no_cpu: bool) -> dict:
    """SURVEY.md 8(f) row 3 at configs[2] size: integrate -> contact model -> cost -> arg-min (+ the
    fused exchange), pose in registers, 48 B (twist) per evaluation from HBM."""
    from bipedal_locomotion_framework_b200.system import RolloutBatch
    torch, batch, dev, syn = cx.torch, cx.batch, cx.dev, cx.syn
    n = planes_np.shape[1]
    chains = FEET * SAMPLES
    first = cx.rank * SAMPLES
    NSETS = 3
    planes = [torch.from_numpy(planes_np).to(dev) for _ in range(NSETS)]
    rb = RolloutBatch(batch)
    calls = [rb.prepare(SAMPLES, FEET, HORIZON, 0.01, 0.01, planes[j][0:6], planes[j][6:9, :chains],
                        planes[j][9:18, :chains], planes[j][18:30, :chains], REF_WRENCH, WEIGHTS, mask=0,
                        index_base=first, want_cost=False) for j in range(NSETS)]
    if cx.peer is not None:
        cx.peer.fuse_into_rollouts(True)

    def step(i):
        call, o = calls[i % NSETS]
        call()
        if cx.world == 1:
            return o["best"]
        if cx.peer is not None:
            return cx.peer.global_best
        return batch.argmin_pairs(cx.sharding.all_gather_pairs(o["best"], cx.world, cx.dist))

    for i in range(W):
        fbest = step(i)
    cx.barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(K):
        fbest = step(i)
    f1.record()
    cx.barrier()
    ms = cx.max_over_ranks(f0.elapsed_time(f1))
    if cx.peer is not None:
        cx.peer.fuse_into_rollouts(False)
    fc, fi = batch.decode_best(fbest)
    res = {"what": "blf_ccm_rollout_integrate_cost at configs[2] size per GPU (weak): ForwardEuler("
                   "FloatingBaseSystemKinematics) -> contact wrench -> cost -> arg-min, cost only; 48 B (twist) "
                   "per evaluation from HBM, pose in registers",
           "value": cx.world * n * K / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / K, "steps": K,
           "rho": 0.01, "dT": 0.01, "argmin": {"cost": fc, "rollout": fi}}
    if cx.world == 1:
        hp = torch.from_numpy(planes_np).pin_memory()
        host_args = (SAMPLES, FEET, HORIZON, 0.01, 0.01, hp[0:6], hp[6:9, :chains], hp[9:18, :chains],
                     hp[18:30, :chains], REF_WRENCH, WEIGHTS)
        for _ in range(3):
            rb.run_host(*host_args, want_cost=False)
        Kh = max(3, min(K, 30))
        t0 = time.perf_counter()
        for _ in range(Kh):
            hb = rb.run_host(*host_args, want_cost=False)
        host_s = (time.perf_counter() - t0) / Kh
        res["e2e"] = {"value": n / host_s, "unit": UNIT, "ms_per_step": host_s * 1e3, "steps": Kh,
                      "h2d_bytes_per_step": int(n * 48 + chains * 24 * 8), "d2h_bytes_per_step": 16,
                      "api": "blf_ccm_rollout_integrate_cost_host (time-major twist planes and per-chain poses "
                             "in pinned host memory in, arg-min pair out)",
                      "argmin": {"cost": hb[0], "rollout": hb[1]}}
        if not no_cpu:
            from oracle import sys_oracle
            cores = os.cpu_count() or 1
            best_s = None
            for _ in range(3):
                t0 = time.perf_counter()
                sys_oracle.rollout(SAMPLES, FEET, HORIZON, 0.01, 0.01, planes_np[0:6], planes_np[6:9, :chains],
                                   planes_np[9:18, :chains], planes_np[18:30, :chains],
                                   uniform=syn.REFERENCE_TEST_PARAMS, mask=0, wrench_ref=REF_WRENCH,
                                   weights=WEIGHTS, nthreads=cores)
                dt_ = time.perf_counter() - t0
                best_s = dt_ if best_s is None else min(best_s, dt_)
            res["cpu_baseline"] = {"value": n / best_s, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": "best of 3 passes of oracle/sys_oracle.c rollout over the same "
                                             "4096 x 2 x 100 batch"}
    return res


def next_rows_leg(cx: Ctx, planes_np, no_cpu: bool = False) -> dict:
    """The rows next to the path, one GPU, briefly (fractions of the measured HBM peak)."""
    from bipedal_locomotion_framework_b200.system import GeneralizedForceBatch, KinematicsBatch
    torch, batch, dev = cx.torch, cx.batch, cx.dev
    n = planes_np.shape[1]
    planes = [torch.from_numpy(planes_np).to(dev) for _ in range(3)]

    def timed(fn, iters=50):
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(iters):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters
    gf = GeneralizedForceBatch(batch)
    rows = {}
    for ncols in (29, 12, 6):                      # 6 + 23 DoF (iCub-sized), and the narrow Jacobians
        cps = FEET
        Js = [torch.rand((n, 6, ncols), dtype=torch.float64, device=dev) for _ in range(2)]
        base = torch.rand((n // cps, ncols), dtype=torch.float64, device=dev)
        gouts = [torch.empty_like(base) for _ in range(2)]
        gcalls = [gf.prepare(cps, ncols, planes[j], Js[j], base, out=gouts[j])[0] for j in range(2)]
        g_ms = timed(lambda i: gcalls[i % 2]())
        g_bytes = n * (200 + 48 * ncols) + (n // cps) * ncols * 16
        rows[f"generalized_force_{ncols}cols"] = {
            "what": f"blf_ccm_generalized_force_soa: base + sum J^T wrench, {n // cps} systems x {cps} contacts, "
                    f"6 x {ncols} Jacobians",
            "ms": g_ms, "contacts_per_s": n / (g_ms * 1e-3), "algorithmic_gbs": g_bytes / (g_ms * 1e-3) / 1e9,
            "hbm_frac_of_measured": g_bytes / (g_ms * 1e-3) / 1e9 / cx.peak}
        del Js, base, gouts, gcalls
    # the end of FloatingBaseDynamicalSystem::dynamics: (M).llt().solve(-h + sum J^T wrench + torques)
    from bipedal_locomotion_framework_b200.system import FloatingBaseDynamicsBatch
    dyn = FloatingBaseDynamicsBatch(batch)
    for ncols in (29, 12):
        cps, ns = FEET, n // FEET
        Ms = []
        for _ in range(2):
            A = torch.rand((ns, ncols, ncols), dtype=torch.float64, device=dev) * 2 - 1
            M = torch.bmm(A, A.transpose(1, 2)) / ncols
            del A
            M.diagonal(dim1=1, dim2=2).add_(0.5)
            Ms.append(M)
        Js = [torch.rand((n, 6, ncols), dtype=torch.float64, device=dev) for _ in range(2)]
        bias = torch.rand((ns, ncols), dtype=torch.float64, device=dev)
        tau = torch.rand((ns, ncols - 6), dtype=torch.float64, device=dev)
        outs = [torch.empty_like(bias) for _ in range(2)]
        scalls = [dyn.prepare_solve(Ms[j], bias, tau, out=outs[j])[0] for j in range(2)]
        s_ms = timed(lambda i: scalls[i % 2](), iters=20)
        acalls = [dyn.prepare_acceleration(cps, planes[j], Js[j], bias, Ms[j], tau, out=outs[j])[0] for j in range(2)]
        a_ms = timed(lambda i: acalls[i % 2](), iters=20)
        # one ForwardEuler step of the whole state with that acceleration (blf_sys_floating_base_euler_step)
        nu, jp = torch.rand_like(bias), torch.rand_like(tau)
        bp = torch.rand((ns, 3), dtype=torch.float64, device=dev)
        br = torch.eye(3, dtype=torch.float64, device=dev).reshape(1, 9).repeat(ns, 1)
        ecall = dyn.prepare_euler_step(0.01, 1e-5, outs[0], nu, jp, bp, br)
        e_ms = timed(lambda i: ecall(), iters=20)
        e_bytes = 8 * (5 * ncols + 12)       # acc in, nu / joints / base pose in and out
        tri = 8 * (ncols * (ncols + 1) // 2 + 2 * ncols + (ncols - 6))       # what LLT reads + rhs in + acc out + torques
        dense = 8 * (ncols * ncols + 2 * ncols + (ncols - 6))                 # the dense matrix the caller hands over
        a_bytes = cps * (200 + 48 * ncols) + tri
        row = {"what": f"blf_sys_mass_matrix_solve / blf_sys_floating_base_acceleration: {ns} systems x {cps} contacts, "
                       f"{ncols} unknowns (6 + {ncols - 6} joints), random symmetric positive definite mass matrices",
               "solve_ms": s_ms, "solve_systems_per_s": ns / (s_ms * 1e-3),
               "solve_hbm_frac_lower_triangle_bytes": ns * tri / (s_ms * 1e-3) / 1e9 / cx.peak,
               "solve_hbm_frac_dense_bytes": ns * dense / (s_ms * 1e-3) / 1e9 / cx.peak,
               "whole_step_ms": a_ms, "whole_step_systems_per_s": ns / (a_ms * 1e-3),
               "hbm_frac_of_measured": ns * a_bytes / (a_ms * 1e-3) / 1e9 / cx.peak,
               "euler_step_ms": e_ms, "euler_step_systems_per_s": ns / (e_ms * 1e-3),
               "euler_step_hbm_frac": ns * e_bytes / (e_ms * 1e-3) / 1e9 / cx.peak,
               "bound": ("HBM on dense bytes (tiles refilled by bulk copies)" if ncols in (6, 8, 12) else
                         "shared-memory data pipe (a third of it the per-thread tile refills) and column-to-column "
                         "latency, not HBM") + " (DESIGN section 10 row 5)"}
        if cx.rank == 0 and not no_cpu:
            from oracle import sys_oracle          # cpu_baseline leg: the C restatement, all host cores
            cores = os.cpu_count() or 1
            sample = 20000
            Mh, kh, th = (x[:sample].cpu().numpy() for x in (Ms[0], bias, tau))
            best_s = None
            for _ in range(3):
                t0 = time.perf_counter()
                sys_oracle.mass_matrix_solve(Mh, kh, th, nthreads=cores)
                dt_ = time.perf_counter() - t0
                best_s = dt_ if best_s is None else min(best_s, dt_)
            row["cpu_baseline"] = {"value": sample / best_s, "unit": "systems/s", "cores": cores, "kind": "port",
                                   "sample": f"best of 3 passes of oracle/sys_oracle.c syso_mass_matrix_solve over "
                                             f"the first {sample} systems"}
        rows[f"floating_base_dynamics_{ncols}"] = row
        del Ms, Js, bias, tau, outs, scalls, acalls, ecall, nu, jp, bp, br
        torch.cuda.empty_cache()
    kb = KinematicsBatch(cx.local, batch.handle)
    kp = [planes[j][6:18].clone() for j in range(3)]
    kcalls = [kb.prepare_euler_step(0.01, 1e-4, planes[j][0:6], kp[j][0:3], kp[j][3:12]) for j in range(3)]
    k_ms = timed(lambda i: kcalls[i % 3]())
    rows["kinematics_euler_step"] = {"what": "blf_sys_kinematics_euler_step_soa, rho 0.01, 240 B/system",
                                     "ms": k_ms, "systems_per_s": n / (k_ms * 1e-3),
                                     "hbm_frac_of_measured": n * 240 / (k_ms * 1e-3) / 1e9 / cx.peak}
    return rows


def e2e_leg(cx: Ctx, K: int) -> dict:
    """The same evaluation through the reference-facing C-ABI call with HOST buffers:
    blf_ccm_eval_batch_host on arrays of iDynTree-layout objects in pinned host memory, host<->device
    copies inside the timed region, E2E_PER_RANK states per rank and step (a bounded sample of the
    workload: 2^28 states in host memory would be 167 GB)."""
    from bipedal_locomotion_framework_b200.contact_models import FULL
    torch, batch, dev, syn = cx.torch, cx.batch, cx.dev, cx.syn
    n = E2E_PER_RANK
    st = syn.make_states(n, seed=46, start=cx.rank * n)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h_tw, h_po, h_nu = pin(st["twists"]), pin(st["poses"]), pin(st["null_poses"])
    h_out = {"wrench": torch.empty((n, 6), dtype=torch.float64).pin_memory(),
             "autodyn": torch.empty((n, 6), dtype=torch.float64).pin_memory(),
             "ctrl": torch.empty((n, 36), dtype=torch.float64).pin_memory(), "regressor": None}
    Ke = max(3, min(K, 10))

    def run(steps):
        cx.barrier()
        l0 = batch.handle.launch_count
        t0 = time.perf_counter()
        for _ in range(steps):
            batch.evaluate_host(h_tw, h_po, h_nu, None, FULL, out=h_out)
        dt = time.perf_counter() - t0
        return cx.max_over_ranks(dt), batch.handle.launch_count - l0

    for _ in range(2):
        batch.evaluate_host(h_tw, h_po, h_nu, None, FULL, out=h_out)
    e2e_s, launches = run(Ke)
    # parity of the host path (compact control-matrix download + host expansion) on a sample
    from oracle import ccm_oracle
    sel = np.arange(0, n, 257)
    sub = {"n": len(sel), "twists": st["twists"][sel], "poses": st["poses"][sel],
           "null_poses": st["null_poses"][sel], "params": None, "uniform": syn.REFERENCE_TEST_PARAMS}
    refo = ccm_oracle.eval_batch_states(sub, mask=7, nthreads=os.cpu_count() or 1)
    worst = 0.0
    for key in ("wrench", "autodyn", "ctrl"):
        g = h_out[key].numpy()[sel]
        den = np.maximum(np.abs(refo[key]).max(axis=1, keepdims=True), 1e-300)
        worst = max(worst, float((np.abs(g - refo[key]) / den).max()))
    zmask = np.ones(36, dtype=bool)
    for q in range(3):
        zmask[6 * q + q] = False
        zmask[6 * (3 + q) + 3: 6 * (3 + q) + 6] = False
    zeros_ok = bool((h_out["ctrl"].numpy()[:, zmask].view(np.int64) == 0).all())
    d2h_compact = n * (12 + 8) * 8
    e2e = {"value": cx.world * n * Ke / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": int(n * 30 * 8), "d2h_bytes_per_step": int(d2h_compact),
           "ms_per_step": e2e_s / Ke * 1e3, "steps": Ke, "launches_per_step": launches / Ke,
           "evals_per_step_per_gpu": n, "scaling": "weak (a fixed host sample per rank)",
           "api": "blf_ccm_eval_batch_host (AoS iDynTree-layout arrays in pinned host memory in/out; the control "
                  "matrix crosses PCIe as its 7 distinct values and is expanded to the dense Matrix6x6 array by "
                  "the library's host threads)",
           "parity": {"sampled_states": int(len(sel)), "worst_rel_err": cx.max_over_ranks(worst),
                      "structural_zeros_exact": cx.min_flag(zeros_ok), "tol": 1e-12,
                      "ok": bool(cx.max_over_ranks(worst) <= 1e-12) and cx.min_flag(zeros_ok)}}
    # A/B: the dense download (384 B/eval back) that the compact transfer replaces
    batch.set_host_threads(0)
    batch.evaluate_host(h_tw, h_po, h_nu, None, FULL, out=h_out)
    dense_s, _ = run(max(2, Ke // 2))
    batch.set_host_threads(-1)
    e2e["dense_download"] = {"value": cx.world * n * max(2, Ke // 2) / dense_s, "unit": UNIT,
                             "d2h_bytes_per_step": int(n * 48 * 8)}
    # what bounds e2e: the PCIe links, measured here with plain pinned copies of the same byte counts in
    # both directions at once on every rank at the same time, no kernel
    d_up = torch.empty(n * 30, dtype=torch.float64, device=dev)
    d_dn = torch.empty(n * 20, dtype=torch.float64, device=dev)
    h_dn = torch.empty(n * 20, dtype=torch.float64).pin_memory()
    h_up = h_out["ctrl"].view(-1)[: n * 30]
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()

    def both():
        with torch.cuda.stream(s_up):
            d_up.copy_(h_up, non_blocking=True)
        with torch.cuda.stream(s_dn):
            h_dn.copy_(d_dn, non_blocking=True)
    for _ in range(2):
        both()
    cx.barrier()
    tp = time.perf_counter()
    for _ in range(5):
        both()
    torch.cuda.synchronize()
    link_s = cx.max_over_ranks((time.perf_counter() - tp) / 5)
    e2e["pcie"] = {"what": f"pinned cudaMemcpyAsync of one step's bytes (240 B up, 160 B down per evaluation) in both "
                           f"directions at once on all {cx.world} ranks at the same time, no kernel, no expansion",
                   "h2d_gbs_per_gpu": n * 240 / link_s / 1e9, "d2h_gbs_per_gpu": n * 160 / link_s / 1e9,
                   "ceiling_evals_per_s": cx.world * n / link_s,
                   "frac_of_ceiling": (cx.world * n * Ke / e2e_s) / (cx.world * n / link_s),
                   "ranks": cx.world}
    return e2e


def run_ours(args):
    cx = Ctx(args)
    torch, syn = cx.torch, cx.syn
    K, W = max(1, args.steps), max(args.warmup, 3)

    head = rollout_workload(
        cx, "configs[4]", HEAD_ROLLOUTS, HEAD_ROLLOUT_LEN, het=False, K=K, W=W, seed=46,
        sustain_s=0.0 if args.only_main else 1.2, force_windows=args.force_windows, dump_dir=args.dump_outputs)
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": cx.world, "steps": K, "warmup": W,
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64",
        "data": "synthetic (device-generated, seeded; the distributions of synthetic.make_states)",
        "config": shared_config(cx.world),
        "layout": "SoA planes in; SoA wrench/autodyn planes + dense row-major 6x6 out",
        "l2": "per-GPU working set (>= 20 GB) >> 126 MB L2: no flush needed",
        "evals_per_step_per_gpu": head["evals_per_step_per_gpu"], "output_windows": head["output_windows"],
        "collective": head["collective"], "collective_note": cx.peer_note,
        "roofline": dict(head["roofline"],
                         kernel="ccm_soa_kernel<WRENCH|AUTODYN|CTRL, uniform, COST> (1 contact/lane, 1 tile/warp) "
                                "+ ccm_cost_reduce_kernel",
                         traffic=None, traffic_bytes_per_eval_ncu=_traffic("ccm_soa_kernel<7,0,1>"),
                         sustained_frac=(head["sustained"] or {}).get("frac")),
        "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "parity": head["parity"],
        "exchange_check": head["exchange_check"], "argmin": head["argmin"], "sustained": head["sustained"],
    }
    tr = line["roofline"]["traffic_bytes_per_eval_ncu"]
    if tr is not None:
        line["roofline"]["traffic"] = tr * head["evals_per_step_per_gpu"]
    torch.cuda.empty_cache()

    if not args.only_main:
        Kx = min(max(K, 10), 200)
        # configs[3]: 64 M heterogeneous states + fused arg-min, strong scaling
        line["configs3_het64m"] = rollout_workload(
            cx, "configs[3]: 64M heterogeneous contact states (per-contact length/width/spring/damper), 335 544 "
                "rollouts of 200 sharded by rollout, wrench+autodyn+ctrl + per-rollout cost + arg-min exchange",
            HET_ROLLOUTS, HET_ROLLOUT_LEN, het=True, K=min(K, 20), W=3, seed=47)
        line["configs3_het64m"]["scaling"] = "strong"
        torch.cuda.empty_cache()
        # configs[2]: per GPU (weak)
        st = syn.make_states(N_MPC, seed=45, start=cx.rank * N_MPC)
        planes_np = syn.aos_to_planes(st["twists"], st["poses"], st["null_poses"])
        c2 = {"eval_only": eval_only_leg(cx, planes_np, max(Kx, 100), 10)}
        c2["mpc"] = rollout_workload(
            cx, "configs[2] per GPU (weak): sampling-MPC batch 2 feet x 4096 samples x 100 steps, wrench+autodyn+"
                "ctrl + per-rollout cost + arg-min exchange",
            cx.world * SAMPLES, MPC_ROLLOUT_LEN, het=False, K=max(Kx, 100), W=10, seed=45, nsets=3,
            host_planes=planes_np)
        c2["mpc"]["scaling"] = "weak"
        c2["mpc_fused"] = fused_rollout_leg(cx, planes_np, max(Kx, 100), 10, args.no_cpu)
        c2["mpc_fused"]["speedup_vs_unfused_mpc"] = c2["mpc"]["ms_per_step"] / c2["mpc_fused"]["ms_per_step"]
        line["configs2"] = c2
        if cx.world == 1:
            line["next_rows"] = next_rows_leg(cx, planes_np, args.no_cpu)
        line["e2e"] = e2e_leg(cx, K)
        line["cpu_baseline"] = None
        if cx.world == 1 and cx.rank == 0 and not args.no_cpu:
            cores = os.cpu_count() or 1
            v, passes, spent, kind, what = cpu_reference_pass(st, cores, min_seconds=3.0)
            cb = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                  "sample": f"best of {passes} passes over a {N_MPC}-state sample of the workload "
                            f"({spent:.1f} s wall x {cores} threads), per-instance path; {what}"}
            if kind == "reference":
                pv, ppasses, _, _, pwhat = cpu_reference_pass(st, cores, 2.0, prefer_reference=False)
                cb["port_value"] = pv
                cb["port_sample"] = f"best of {ppasses} passes, {pwhat}"
            # SURVEY.md 8(d): the same path on ONE thread beside the all-cores figure
            n1 = N_MPC // 8
            st1 = {k: (v[:n1] if hasattr(v, "shape") and v.shape[:1] == (N_MPC,) else v) for k, v in st.items()}
            st1["n"] = n1
            v1, p1, _, _, _ = cpu_reference_pass(st1, 1, min_seconds=1.0)
            cb["single_thread_value"] = v1
            cb["single_thread_sample"] = f"best of {p1} passes over the first {n1} states of that sample, 1 thread"
            line["cpu_baseline"] = cb
    if cx.rank == 0:
        emit(line)
    cx.close()
    return 0


def run_config2(args):
    """BASELINE.json configs[1]: 2^20 states per GPU, wrench only (248 B/eval), run on request."""
    from bipedal_locomotion_framework_b200.contact_models import WRENCH
    cx = Ctx(args)
    torch, syn, batch, dev = cx.torch, cx.syn, cx.batch, cx.dev
    n, nsets = 1 << 20, 3
    K, W = max(1, args.steps), max(min(args.warmup, 10), 3)
    planes, _ = syn.make_planes_torch(n, dev, seed=43 + 1000 * cx.rank)
    sets = [(planes, batch.alloc_soa_outputs(n, WRENCH))] + \
        [([None if q is None else q.clone() for q in planes], batch.alloc_soa_outputs(n, WRENCH))
         for _ in range(nsets - 1)]
    calls = [batch.prepare_soa(pl, None, WRENCH, out=o)[0] for pl, o in sets]
    for i in range(W):
        calls[i % nsets]()
    cx.barrier()
    l0 = batch.handle.launch_count
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        calls[i % nsets]()
    e1.record()
    cx.barrier()
    t1 = time.perf_counter()
    my_ms = e0.elapsed_time(e1)
    ms = cx.max_over_ranks(my_ms)
    from oracle import ccm_oracle
    pl, out = sets[(K - 1) % nsets]
    idx = torch.arange(0, n, 17, device=dev)
    stt = syn.sample_states_from_planes(pl, None, idx)
    refo = ccm_oracle.eval_batch_states(stt, mask=1, nthreads=os.cpu_count() or 1)
    got = torch.stack([p[idx] for p in out["wrench"]], 1).cpu().numpy()
    worst = 0.0
    for sl in (slice(0, 3), slice(3, 6)):
        num = np.abs(got[:, sl] - refo["wrench"][:, sl]).max(axis=1)
        den = np.maximum(np.abs(refo["wrench"][:, sl]).max(axis=1), 1e-300)
        worst = max(worst, float(np.where(num == 0, 0, num / den).max()))
    gbs = 248 * n / (my_ms / K * 1e-3) / 1e9
    if cx.rank == 0:
        emit({"metric": METRIC, "value": cx.world * n * K / (ms * 1e-3), "unit": UNIT, "n_gpus": cx.world,
              "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
              "vs_baseline": None, "dtype": "f64", "data": "synthetic (device-generated)",
              "config": {"workload": "configs[1]: 1M random contact states per GPU, wrench only, uniform foot geometry "
                                     "and stiffness/damping, SoA (25 live planes in, 6 planes out = 248 B/eval)",
                         "evals_per_step": cx.world * n,
                         "l2": "3 rotating input/output buffer sets; one step streams 260 MB (> 126 MB L2)"},
              "roofline": {"bound": "hbm", "achieved": gbs, "peak": cx.peak, "unit": "GB/s", "frac": gbs / cx.peak,
                           "traffic": None, "peak_source": cx.peak_src},
              "cpu_baseline": None, "e2e": None, "gpu_launches": int(batch.handle.launch_count - l0),
              "clocks": cx.sampler.summary(t0, t1),
              "parity": {"sampled_states": int(idx.numel()), "worst_block_rel_err": worst, "tol": 1e-12,
                         "ok": bool(worst <= 1e-12)}})
    cx.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="headline", choices=["headline", "config2"],
                    help="headline (default): configs[4] strong scaling as `value` + configs[3], configs[2], e2e, "
                         "cpu_baseline records; config2: configs[1], 1M states wrench-only")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--nccl-argmin", action="store_true",
                    help="N > 1: use the NCCL all-gather for the arg-min pair instead of the "
                         "peer-memory mailbox")
    ap.add_argument("--only-main", action="store_true",
                    help="profiling aid: run only the headline timed loop (no extra records)")
    ap.add_argument("--force-windows", type=int, default=0,
                    help="testing aid: reuse an output window of 1/W of the shard (the low-memory fallback)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="headline workload: write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "ours" or args.workload != "headline"):
        ap.error("--dump-outputs applies to the headline workload of --impl ours")
    # stdout carries exactly ONE JSON line: whatever libraries print there (NCCL's version banner
    # when NCCL_DEBUG is set on the box) is sent to stderr at the file-descriptor level
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "config2":
        return run_config2(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
