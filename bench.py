#!/usr/bin/env python
"""Benchmark of the batched whole-body QP control step (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (dynamics + ID-QP: the reduce kernel and the solve kernel, stream ordered; a 4096-65536
instance batch goes through as 2-4 chunks of that pair on as many streams, forked from and joined to the launch stream, so
`gpu_launches` is 4 per step at 4096) over one batch of synthetic states.
Workload at N = 1: BASELINE.json configs[1] - mini_cheetah ID-QP, 4096 random states per launch, all four feet in stance
(SURVEY.md 8d). With N > 1 (torchrun, one rank per GPU) every rank runs the same batch size on its own shard of instances
(weak scaling, no collective on the data path); `--total T` instead splits T instances over the ranks (strong scaling,
BASELINE configs[4]).

Printed JSON (rank 0): value = control steps/s with inputs resident in HBM (CUDA events on the launch stream, L2 flushed
between timed launches, max over ranks); e2e = the same through `wbc_step_host` with pinned host buffers (H2D + kernels +
D2H inside the timed region); roofline / cpu_baseline as the contract asks; latency_n1 = p50 of ONE control step of ONE
robot through the LeafSystem mirror (the reference's operating point: one step per 5 ms, simulate.py:20-22).
`--impl reference` times the CPU restatement of the reference path (oracle/, C port) on the host cores instead - pydrake /
OSQP themselves are not installable (DESIGN.md 5); `import pydrake` is probed at start and reported either way.
`--dump-outputs DIR` writes the outputs of the last timed step as DIR/<name>.npy; with N > 1 these are rank 0's shard only,
so two builds are compared on that shard.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

ROBOT, PATTERN, BATCH, SEED = "mini_cheetah", "stand", 4096, 20260119
METRIC = "whole-body QP control steps/sec"
ALGO_BYTES_PER_STEP = 860          # SURVEY 8d: q,v 296 + traj 432 + contact 4 in; tau 96 + metrics 32 out
CANON_FLOPS_PER_STEP = {0: 0.56e6, 1: 0.78e6, 2: 1.05e6, 3: 1.37e6, 4: 1.75e6}   # SURVEY 8d F(nc) @ 12 IPM iterations
WORKLOAD = "mini_cheetah ID-QP controller step, 4096 random synthetic states (BASELINE configs[1])"


def shared_config(args, n_per_gpu, world):
    """The workload description both arms print, key for key (the driver compares them)."""
    total = n_per_gpu * world
    experiment = (n_per_gpu != BATCH or args.pattern != PATTERN or args.robot != ROBOT or args.controller != "id" or args.torque_limits
                  or args.total)
    wl = WORKLOAD if not experiment else (
        f"EXPERIMENT (not the BASELINE bench config): {args.robot} {args.controller.upper()}-QP, {n_per_gpu} instances/launch/GPU, "
        f"pattern {args.pattern}, torque limits {'on' if args.torque_limits else 'off'}")
    return {"workload": wl, "robot": args.robot, "controller": args.controller.upper(), "contact_pattern": args.pattern,
            "instances_per_step_per_gpu": int(n_per_gpu), "torque_limits": bool(args.torque_limits), "seed": SEED,
            "tie_break_reg_f": 1e-6, "total_instances": int(total) if args.total else None}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def flop_model():
    """Executed FP64 work per instance as a function of the measured active-set iterations. STATIC: fitted to ncu captures
    of this kernel build (tools/ncu_flops.py -> profiles/r2_flop_model.json); the file names the captures and the commit."""
    p = ROOT / "profiles" / "r2_flop_model.json"
    return json.loads(p.read_text()) if p.exists() else None


DUMP_MAX_ROWS = 1 << 18             # 5 float64 files of 22 columns in all: 176 B a row, 46 MB at this cap


def dump_rows(n):
    """Instances written by --dump-outputs: the whole batch, or above DUMP_MAX_ROWS a fixed seeded sample (sorted)."""
    if n <= DUMP_MAX_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(SEED).choice(n, DUMP_MAX_ROWS, replace=False))


def dump_outputs(out_dir, n, outputs):
    """Writes the device outputs of the last timed step as out_dir/<name>.npy (float64; status codes and the row indices
    in rows.npy are exact in float64), so that two builds run with the same arguments can be compared output for output."""
    import torch
    rows = dump_rows(n)
    idx = torch.from_numpy(rows).to(next(iter(outputs.values())).device)
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "rows.npy", rows.astype(np.float64))
    for name, t in outputs.items():
        np.save(d / f"{name}.npy", t.index_select(0, idx).cpu().numpy().astype(np.float64))


class ClockSampler:
    """SM clock and throttle reasons while the GPU is under this benchmark's load, polled through NVML from a thread.
    It runs from the first warm-up launch to the last timed launch (the timed region alone lasts ~2 ms at --steps 20, too
    short for more than one NVML sample); `in_timed` counts the samples that fell inside the timed region."""

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz, self.err = index, [], set(), None, None
        self._stop = threading.Event()
        self._th = None
        self.timed = False
        self.in_timed = 0

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].strip().isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            return
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                if self.timed:
                    self.in_timed += 1
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = int(get(self.h))
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                break
            time.sleep(0.001)

    def stop(self):
        self._stop.set()
        if self._th is not None:
            self._th.join(timeout=2.0)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
               "reasons": sorted(self.reasons), "samples": len(self.sm), "samples_in_timed_region": self.in_timed,
               "source": "NVML polled every ~1 ms from the first warm-up launch to the last timed launch"}
        if self.err:
            out["error"] = self.err
        return out


# ------------------------------------------------------------------------------- CPU arm
def cpu_port_throughput(robot, q, v, traj, contact, budget_s=20.0, single_thread_s=3.0, **params):
    """C port of the oracle (CPU restatement of the reference path, NOT Drake + OSQP) on all host cores + one thread. It
    solves the reference QP as the reference builds it: the optional torque box (not in the reference) is not part of it."""
    from oracle.cport import time_id_steps
    return time_id_steps(robot, q, v, traj, contact, budget_s, single_thread_s)


def run_reference(args):
    """Reference arm: the CPU restatement of the reference path (C twin of the oracle, gcc -O3 -march=native) on all host
    cores, same config / metric / unit; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import __graft_entry__ as g
    g.build_oracle()
    from quadruped_drake_b200 import drake_bridge, load_robot
    from quadruped_drake_b200.synth import generate
    from oracle.cport import fk as cfk
    if args.controller != "id":
        raise SystemExit("bench.py --impl reference: the timed C port covers the ID controller (the BASELINE bench config)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n = args.total // world if args.total else args.batch
    model = load_robot(args.robot)
    ns = min(n, 4096)                                           # bounded sample of the batch (the same first instances)
    q, v, traj, contact = generate(model, ns, SEED, args.pattern, cfk(args.robot))
    vals = []
    per_step = max(2.0, min(20.0, 120.0 / (args.warmup + args.steps)))
    extra = {"torque_limits": 1} if args.torque_limits else {}
    for s in range(args.warmup + args.steps):
        last = s == args.warmup + args.steps - 1                  # the single-thread figure is taken once, on the last step
        r = cpu_port_throughput(args.robot, q, v, traj, contact, budget_s=per_step, single_thread_s=3.0 if last else 0.0, **extra)
        if s >= args.warmup:
            vals.append(r)
    val = float(np.mean([r["value"] for r in vals]))
    base = dict(vals[-1])
    base["value"] = val
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * n / val, "higher_is_better": True,
            "scaling": "strong" if args.total else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": shared_config(args, n, world),
            "reference_kind": "CPU restatement of the reference path (C port of the oracle), NOT Drake + OSQP: pydrake is not "
                              "installable here (DESIGN.md 5); each step is a bounded sample of the batch on all host cores",
            "pydrake": drake_bridge.probe(),
            "cpu_baseline": base,
            "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------- GPU arm
def latency_n1(ctl_kwargs, robot, device):
    """p50 latency of one control step of one robot: (a) IDController.DoSetControlTorques through the LeafSystem mirror
    (EvalOutput of "quad_torques", SimpleStanding input: BASELINE configs[0]); (b) wbc_step_host with N = 1 on page-locked
    buffers; (c) the device-resident step (CUDA events). The reference runs this once per 5 ms (simulate.py:20-22)."""
    import ctypes as C
    import torch
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200.controller import IDController
    from quadruped_drake_b200.planner import BasicTrunkPlanner
    leaf = IDController(robot, 5e-3, device=device, **ctl_kwargs)
    planner = BasicTrunkPlanner(robot=robot)
    q0 = leaf.batched.model.nominal_q()
    ctx = leaf.CreateDefaultContext()
    ctx.FixValue(0, np.hstack([q0, np.zeros(18)]))
    ctx.FixValue(1, planner.SetTrunkOutputs(0.0))
    for _ in range(20):
        leaf.EvalOutput(ctx, 0)
    ts = []
    for _ in range(300):
        t0 = time.perf_counter()
        leaf.EvalOutput(ctx, 0)
        ts.append(time.perf_counter() - t0)
    out = {"leafsystem_p50_us": 1e6 * float(np.median(ts)), "leafsystem_p99_us": 1e6 * float(np.percentile(ts, 99))}
    ctl = leaf.batched
    from quadruped_drake_b200.controller import dict_to_traj
    traj, contact = dict_to_traj(planner.SetTrunkOutputs(0.0))
    hq, hv, ht = capi.pinned_empty((1, 19)), capi.pinned_empty((1, 18)), capi.pinned_empty((1, 54))
    hc = capi.pinned_empty((1, 4), np.uint8)
    hq[:], hv[:], ht[:], hc[:] = q0, 0.0, traj, contact
    htau, hmet, hst = capi.pinned_empty((1, 12)), capi.pinned_empty((1, 4)), capi.pinned_empty((1,), np.int32)
    hio = capi.WbcIO(capi.np_ptr(hq), capi.np_ptr(hv), capi.np_ptr(ht), capi.np_ptr(hc), capi.np_ptr(htau), capi.np_ptr(hmet),
                     capi.np_ptr(hst))
    for _ in range(20):
        ctl.lib.wbc_step_host(ctl._h, capi.WBC_CTRL_ID, 1, C.byref(hio))
    ts = []
    for _ in range(300):
        t0 = time.perf_counter()
        ctl.lib.wbc_step_host(ctl._h, capi.WBC_CTRL_ID, 1, C.byref(hio))
        ts.append(time.perf_counter() - t0)
    out["step_host_p50_us"] = 1e6 * float(np.median(ts))
    dev = torch.device(f"cuda:{device}")
    tq, tv, tt = (torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (hq, hv, ht))
    tc = torch.from_numpy(np.ascontiguousarray(hc)).to(dev)
    tau = torch.empty((1, 12), dtype=torch.float64, device=dev)
    met = torch.empty((1, 4), dtype=torch.float64, device=dev)
    st = torch.empty((1,), dtype=torch.int32, device=dev)
    io = ctl.make_io(tq, tv, tt, tc, tau, met, st)
    stream = torch.cuda.current_stream(dev)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(100)]
    for _ in range(10):
        ctl.lib.wbc_step(ctl._h, capi.WBC_CTRL_ID, 1, C.byref(io), C.c_void_p(stream.cuda_stream))
    for e0, e1 in evs:
        e0.record(stream)
        ctl.lib.wbc_step(ctl._h, capi.WBC_CTRL_ID, 1, C.byref(io), C.c_void_p(stream.cuda_stream))
        e1.record(stream)
    torch.cuda.synchronize()
    out["device_step_p50_us"] = 1e3 * float(np.median([e0.elapsed_time(e1) for e0, e1 in evs]))
    out["status"] = int(hst[0])
    # BASELINE configs[0]: the reference's whole simulate.py loop for one robot (planner -> controller ports -> plant step)
    try:
        sys.path.insert(0, str(ROOT / "examples"))
        import simulate
        simulate.run("id", "standing", sim_time=0.25, verbose=False)
        t0 = time.perf_counter()
        _, _, lg = simulate.run("id", "standing", sim_time=2.0, verbose=False)
        out["simulate_loop_steps_per_s"] = len(lg) / getattr(simulate.run, "last_wall", time.perf_counter() - t0)   # the loop itself
        out["simulate_loop_note"] = ("examples/simulate.py: BasicTrunkPlanner -> IDController (LeafSystem mirror) -> wbc_plant_step, one robot, dt 5e-3; "
                                     "the reference's Drake loop ran at ~180-200 steps/s (BASELINE.md 1)")
    except Exception as e:  # noqa: BLE001
        out["simulate_loop_error"] = repr(e)
    out["reference_period_us"] = 5000.0
    out["note"] = ("one robot, one control step: launch -> torques in host memory; the reference's own loop ran at ~180-200 "
                   "steps/s including the plant step (BASELINE.md 1)")
    leaf.batched.close()
    return out


def run_gpu(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the controller path has no CPU fallback (use --impl reference for the CPU arm)")
    if rank == 0:
        g.build()
    if world > 1:
        # NCCL announces its version on stdout when the first communicator comes up; stdout carries only the JSON line, so
        # it is pointed at stderr for the rendezvous
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    from quadruped_drake_b200 import capi, drake_bridge
    from quadruped_drake_b200.controller import BatchedController, measure_fp64_peak
    from quadruped_drake_b200.sharding import shard_range
    from quadruped_drake_b200.synth import generate

    robot = args.robot
    kind = capi.KINDS[args.controller]
    ctl_kwargs = {"torque_limits": 1} if args.torque_limits else {}
    ctl = BatchedController(robot, device=local, **ctl_kwargs)
    if args.total:                                              # strong scaling: contiguous shard of [0, total)
        lo, hi = shard_range(args.total, rank, world)
        n = hi - lo
    else:
        n = args.batch
    # every rank its own shard of instances; generated in pieces so that 10^7 instances do not need 10^7-row FK temporaries
    parts = [generate(ctl.model, min(1 << 20, n - o), SEED + 1000 * rank + 17 * (o >> 20), args.pattern, ctl.fk) for o in range(0, n, 1 << 20)]
    q, v, traj, contact = (np.concatenate([p[i] for p in parts]) for i in range(4))
    del parts
    tq, tv, tt = (torch.from_numpy(x).to(dev) for x in (q, v, traj))
    tc = torch.from_numpy(contact).to(dev)
    tau = torch.empty((n, 12), dtype=torch.float64, device=dev)
    met = torch.empty((n, 4), dtype=torch.float64, device=dev)
    st = torch.empty((n,), dtype=torch.int32, device=dev)
    qi = torch.empty((n, 4), dtype=torch.float64, device=dev)
    io = ctl.make_io(tq, tv, tt, tc, tau, met, st, None, None, qi)
    stream = torch.cuda.current_stream(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)       # 256 MB > 126 MB L2

    def launch():
        rc = ctl.lib.wbc_step(ctl._h, kind, n, C.byref(io), C.c_void_p(stream.cuda_stream))
        if rc:
            raise RuntimeError(ctl.lib.wbc_last_error(ctl._h).decode())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        flush.zero_()
        launch()
    torch.cuda.synchronize()
    status = st.cpu().numpy()
    iters = float(qi[:, 3].mean().item())
    iters_max = float(qi[:, 3].max().item())
    bad = status != 0
    if args.controller in ("pc", "mptc"):
        bad &= status != capi.ST_UNSUPPORTED          # full-flight instances: the reference PC / MPTC raise there too (SURVEY E.5c)
    if bad.mean() > (1e-3 if args.torque_limits else 0.0):
        raise SystemExit(f"bench.py: {int(bad.sum())} of {n} instances returned a non-zero status")

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = ctl.launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler.timed = True
    for e0, e1 in evs:
        flush.zero_()                       # L2 flush between timed launches (not inside the event pair)
        e0.record(stream)
        launch()
        e1.record(stream)
    torch.cuda.synchronize()
    sampler.timed = False
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, {"tau": tau, "metrics": met, "status": st, "qp_info": qi})
    if world > 1:
        dist.barrier()
    gpu_launches = ctl.launches - launches0
    per = np.array([e0.elapsed_time(e1) for e0, e1 in evs])     # ms per launch
    total_ms = float(per.sum())
    my_ms = total_ms
    per_rank = None
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        # per-rank record (to attribute multi-GPU losses): ms per step, p50, mean / max iterations, instances
        mine = torch.tensor([my_ms / args.steps, float(np.median(per)), iters, iters_max, float(n)], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": r, "ms_per_step": float(a[0]), "p50_ms": float(a[1]), "mean_iterations": float(a[2]),
                     "max_iterations": float(a[3]), "instances": int(a[4])} for r, a in enumerate(allr)]
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel share of the step (events between the two kernels; separate short run, same inputs)
    ms_r, ms_s = C.c_double(), C.c_double()
    shares = None
    if n <= 262144 and ctl.lib.wbc_profile_step(ctl._h, kind, n, C.byref(io), 20, C.c_void_p(stream.cuda_stream), C.byref(ms_r), C.byref(ms_s)) == 0:
        shares = {"reduce_kernel_ms": ms_r.value, "solve_kernel_ms": ms_s.value,
                  "solve_share": ms_s.value / max(ms_r.value + ms_s.value, 1e-12)}

    # ---- end to end through the host API: pinned host buffers, H2D + kernel + D2H every step
    h2d = n * (19 + 18 + 54) * 8 + n * 4
    d2h = n * (12 + 4) * 8 + n * 4
    e2e_s, e2e_steps, e2e_plan = None, 0, None
    if not args.no_e2e:
        hq, hv, ht = capi.pinned_empty((n, 19)), capi.pinned_empty((n, 18)), capi.pinned_empty((n, 54))
        hc = capi.pinned_empty((n, 4), np.uint8)
        hq[:], hv[:], ht[:], hc[:] = q, v, traj, contact
        htau, hmet, hst = capi.pinned_empty((n, 12)), capi.pinned_empty((n, 4)), capi.pinned_empty((n,), np.int32)
        hio = capi.WbcIO(capi.np_ptr(hq), capi.np_ptr(hv), capi.np_ptr(ht), capi.np_ptr(hc), capi.np_ptr(htau), capi.np_ptr(hmet),
                         capi.np_ptr(hst), None, None, None)
        for _ in range(3):
            ctl.lib.wbc_step_host(ctl._h, kind, n, C.byref(hio))
        if world > 1:
            dist.barrier()
        e2e_steps = args.steps if n <= (1 << 20) else max(3, args.steps // 4)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            rc = ctl.lib.wbc_step_host(ctl._h, kind, n, C.byref(hio))
            assert rc == 0
        e2e_s = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        assert np.array_equal(htau, tau.cpu().numpy()), "host and device entry points disagree"
        h2d = n * (19 + 18 + 54) * 8 + n * 4
        d2h = n * (12 + 4) * 8 + n * 4
        # ---- second end-to-end figure: trunk targets from a device-resident plan (the host sends q, v, t only: 308 B / instance)
        e2e_plan = None
        if world == 1 and (not args.no_cpu or args.plan) and kind != capi.WBC_CTRL_PD and n <= (1 << 20):
            try:
                from quadruped_drake_b200 import planner as pl
                bh = float(ctl.model.nominal_q()[6])
                sampler = pl.TrajectorySampler(ctl, [pl.make_motion_plan(robot, m, 6.0, base_height=bh) for m in ("standing", "orientation", "heave")])
                rng = np.random.default_rng(SEED)
                ht_, hpi = capi.pinned_empty((n,)), capi.pinned_empty((n,), np.int32)
                ht_[:], hpi[:] = rng.uniform(0.0, 6.0, n), rng.integers(0, 3, n)
                hq2 = capi.pinned_empty((n, 19))
                hq2[:] = q
                hq2[:, 4:6] = 0.0                                    # the test motions stay over the origin
                for _ in range(3):
                    ctl.step_plan(kind, sampler, hq2, hv, ht_, hpi, htau, hmet, hst)
                okp = float((hst == 0).mean())
                t0 = time.perf_counter()
                for _ in range(e2e_steps):
                    ctl.step_plan(kind, sampler, hq2, hv, ht_, hpi, htau, hmet, hst)
                dtp = time.perf_counter() - t0
                # the same workload through the raw-buffer entry (trajectory rows sampled once, then sent every step): the A/B
                o = sampler.sample(np.asarray(ht_), np.asarray(hpi))
                ht2, hc2 = capi.pinned_empty((n, 54)), capi.pinned_empty((n, 4), np.uint8)
                ht2[:], hc2[:] = o["traj"], o["contact"]
                hio2 = capi.WbcIO(capi.np_ptr(hq2), capi.np_ptr(hv), capi.np_ptr(ht2), capi.np_ptr(hc2), capi.np_ptr(htau), capi.np_ptr(hmet),
                                  capi.np_ptr(hst), None, None, None)
                for _ in range(3):
                    ctl.lib.wbc_step_host(ctl._h, kind, n, C.byref(hio2))
                t0 = time.perf_counter()
                for _ in range(e2e_steps):
                    ctl.lib.wbc_step_host(ctl._h, kind, n, C.byref(hio2))
                dtr = time.perf_counter() - t0
                e2e_plan = {"value": n * e2e_steps / dtp, "unit": "steps/s", "h2d_bytes_per_step": n * (19 + 18 + 1) * 8 + n * 4, "d2h_bytes_per_step": d2h,
                            "solved_fraction": okp, "raw_buffers_same_workload": n * e2e_steps / dtr,
                            "path": "wbc_step_plan_host: q, v, t and the plan index cross the host link, the 54-double trajectory row is sampled on the "
                                    "device from a resident plan (wbc_sample_trajectory -> step kernels); trunk targets = the reference's manual test "
                                    "motions (planners/simple.py:87-115) at random phases, states = the benchmark's random states"}
            except Exception as e:  # noqa: BLE001
                e2e_plan = {"error": repr(e)}
    n_total = n
    gather = None
    if world > 1:
        t = torch.tensor([float(n)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        n_total = int(t.item())
        # the optional gather of the torque shards onto rank 0 over NCCL (SURVEY 8e) - outside the timed region, timed on its own
        from quadruped_drake_b200.sharding import gather_rows
        if n_total * 96 <= (4 << 30):
            gather_rows(tau, n_total, dst=0)
            torch.cuda.synchronize()
            dist.barrier()
            g0 = time.perf_counter()
            full = gather_rows(tau, n_total, dst=0)
            torch.cuda.synchronize()
            gather = {"ms": 1e3 * (time.perf_counter() - g0), "bytes": n_total * 96, "backend": "nccl",
                      "rows_on_rank0": int(full.shape[0]) if full is not None else None}
            del full

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = n_total * args.steps / (total_ms * 1e-3)
    kernel_ms = float(per.mean())
    hbm_peak, peak_src = measured_peaks()
    ach_gbs = ALGO_BYTES_PER_STEP * n / (kernel_ms * 1e-3) / 1e9
    fp64_peak = measure_fp64_peak(local)
    fm = flop_model()
    nc_mean = float(contact.sum(axis=1).mean())
    canon = CANON_FLOPS_PER_STEP[4]
    if fm:
        flops_inst = fm["reduce_flops"] + fm["solve_flops_base"] + fm["solve_flops_per_iteration"] * iters
        traffic = fm.get("dram_bytes_per_instance_4096", 0.0) * n if fm.get("dram_bytes_per_instance_4096") else None
    else:
        flops_inst, traffic = None, None
    ach_tf = (flops_inst or 0.0) * n / (kernel_ms * 1e-3) / 1e12
    cfg = shared_config(args, args.batch if not args.total else args.total // world, world)
    line = {
        "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": total_ms / args.steps, "p50_ms_per_step": float(np.median(per)), "higher_is_better": True,
        "scaling": "strong" if args.total else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "gpu_details": {"l2": "flushed between timed launches (256 MB memset outside the event pair)",
                        "mean_active_set_iterations": iters, "max_active_set_iterations": iters_max,
                        "mean_stance_feet": nc_mean, "kernels": shares, "per_rank": per_rank},
        "e2e": {"value": n_total * e2e_steps / e2e_s if e2e_s else None, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps,
                "path": "wbc_step_host on page-locked host buffers, inputs and outputs cross the host link inside the timed region: the kernels "
                        "read / write host memory directly (zero-copy, below 131072 instances per call) or the batch goes through the "
                        "65536-instance two-stream copy / compute pipeline (above; also the path of pageable buffers)"},
        "e2e_device_plan": e2e_plan,
        "tau_gather": gather,
        "gpu_launches": int(gpu_launches),
        "clocks": clocks,
        "pydrake": drake_bridge.probe(),
        "roofline": {"bound": "fp64", "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach_tf / fp64_peak if fp64_peak else None,
                     "traffic": traffic,
                     "peak_source": "DFMA loop measured in this run (wbc_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
                     "flops_per_step": flops_inst,
                     "basis": ("EXECUTED FP64 work per instance = reduce + solve_base + solve_per_iteration x the mean active-set iterations "
                               "MEASURED in this run; the three coefficients are STATIC, fitted to ncu captures of this kernel build: "
                               + (fm["source"] if fm else "no model file")),
                     "hbm": {"achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak, "peak_source": peak_src,
                             "algorithmic_bytes_per_step": ALGO_BYTES_PER_STEP,
                             "note": "860 B/step of algorithmic I/O: two orders of magnitude below the HBM roof - this path is not HBM bound"},
                     "binding_resource": (fm or {}).get("binding_resource"),
                     "canonical": {"flops_per_step": canon, "tflops_equivalent": canon * n / (kernel_ms * 1e-3) / 1e12,
                                   "note": "SURVEY 8d F(nc=4): 12 interior-point iterations on the reference-size KKT system. The "
                                           "null-space + active-set kernel reaches the exact optimum with ~14x fewer flops, so this "
                                           "equivalent rate can exceed the hardware peak"}},
    }
    if world == 1 and not args.no_cpu:
        ns = min(n, 4096)
        line["cpu_baseline"] = cpu_port_throughput(robot, q[:ns], v[:ns], traj[:ns], contact[:ns], **ctl_kwargs)
        try:
            line["latency_n1"] = latency_n1(ctl_kwargs, robot, local)
        except Exception as e:  # noqa: BLE001
            line["latency_n1"] = {"error": repr(e)}
        if not args.no_aux:
            # rows next to the step (SURVEY 8 f1-f3), short runs: LCM wire codecs, trajectory sampler, closed-loop rollouts
            try:
                sys.path.insert(0, str(ROOT / "tools"))
                import bench_aux
                line["aux"] = bench_aux.summary()
            except Exception as e:  # noqa: BLE001
                line["aux"] = {"error": repr(e)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="instances per launch per GPU (default: the BASELINE config, 4096)")
    ap.add_argument("--total", type=int, default=0, help="strong scaling: total instances, split evenly over the ranks (BASELINE configs[4])")
    ap.add_argument("--pattern", default=PATTERN, choices=["stand", "trot", "walk", "mixed"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and latency legs (experiments only)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (sweeps at 10^7 instances: 8.6 GB of pinned buffers)")
    ap.add_argument("--plan", action="store_true", help="measure `e2e_device_plan` even with --no-cpu")
    ap.add_argument("--no-aux", action="store_true", help="skip the short wire / sampler / rollout measurements of the `aux` key")
    ap.add_argument("--robot", default=ROBOT, choices=["mini_cheetah", "anymal_b"], help="experiments only")
    ap.add_argument("--controller", default="id", choices=["id", "clf", "pc", "mptc"], help="experiments only")
    ap.add_argument("--torque-limits", action="store_true", help="experiments only: |tau| <= effort rows (BASELINE configs[2])")
    ap.add_argument("--workload", default="step", choices=["step", "wire", "traj", "rollout"],
                    help="step = the BASELINE metric (default); wire / traj / rollout = the rows next to it (tools/bench_aux.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps write what the last one computed (tau, metrics, "
                    "status, qp_info of rank 0's batch, or a fixed seeded sample of at most %d instances, listed in rows.npy) "
                    "as DIR/<name>.npy, e.g. DIR = bench_outputs/" % DUMP_MAX_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "step"):
        ap.error("--dump-outputs writes the outputs of the GPU control step (--impl ours --workload step)")
    if args.workload != "step":
        import __graft_entry__ as g
        g.build()
        sys.path.insert(0, str(ROOT / "tools"))
        import bench_aux
        bench_aux.run(args.workload, steps=args.steps, warmup=args.warmup)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
