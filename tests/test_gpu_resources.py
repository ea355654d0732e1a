"""Ownership of the library's device resources: destroying a handle, a plan or a multi-device handle frees everything it
allocated, whatever path grew it, and a plan may be destroyed after the handle it was created with.

Device memory is read per process from NVML, not from cudaMemGetInfo: free memory of the whole device moves with every other
process on it. The first create -> use -> destroy cycle absorbs what the process keeps for good (modules loaded on first
launch, the local-memory reservation of the kernels); a second identical cycle must leave the process where the first did.
NVML counts whole 2 MiB pages, so a leak shows once it spans one: any staging or hand-over buffer of these sizes does, the
few kilobytes of a plan's tables do not."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
BASE = 4096
N_DEV = 8192                         # wbc_step on device buffers: four chains, hand-over slots 0-3
N_PAGEABLE, N_STAGED = 4096, 32768   # wbc_step_host: pageable, then page-locked through staging arrays that must grow
N_PLAN = 4096                        # wbc_step_plan_host: two halves when page-locked
N_SMALL = 256                        # debug / codec entries, rollouts, the multi-device step
Q0 = np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.3] + [0.0, -0.8, 1.6] * 4)


def process_device_bytes():
    """Device memory NVML attributes to this process, summed over the devices; None when NVML does not list the process."""
    pynvml = pytest.importorskip("pynvml")
    pynvml.nvmlInit()
    try:
        used = None
        for i in range(pynvml.nvmlDeviceGetCount()):
            for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i)):
                if p.pid == os.getpid() and p.usedGpuMemory is not None:
                    used = (used or 0) + p.usedGpuMemory
        return used
    finally:
        pynvml.nvmlShutdown()


def rows(base, n):
    idx = np.arange(n) % BASE
    return [np.ascontiguousarray(a[idx]) for a in base]


def motion_plan(ctl):
    from quadruped_drake_b200 import planner as pl
    return pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=float(ctl.model.nominal_q()[6]))


def test_plan_destroyed_after_its_handle(built):
    """A plan keeps no pointer to its handle: destroying it afterwards frees its tables on its device, and the device keeps
    working."""
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    ctl = BatchedController("mini_cheetah", device=0)
    s = pl.TrajectorySampler(ctl, [motion_plan(ctl)])
    ctl.close()
    s.close()
    ctl = BatchedController("mini_cheetah", device=0)
    s = pl.TrajectorySampler(ctl, [motion_plan(ctl)])
    o = s.sample(np.linspace(0.0, 6.0, 64))
    assert (o["status"] == 0).all() and np.isfinite(o["traj"]).all()
    s.close()
    ctl.close()


@pytest.fixture(scope="module")
def inputs(built):
    """Host and device inputs of one cycle, all allocated here: the torch caching allocator must not grow during the cycles."""
    import torch
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.synth import generate
    ctl = BatchedController("mini_cheetah", device=0)
    base = generate(ctl.model, BASE, 11, "mixed", ctl.fk)
    ctl.close()
    d = {"base": base}
    cuda = lambda a: torch.from_numpy(a).to("cuda:0")  # noqa: E731
    q, v, traj, contact = (cuda(a) for a in rows(base, N_DEV))
    f64 = lambda *shape: torch.empty(shape, dtype=torch.float64, device="cuda:0")  # noqa: E731
    d["dev"] = [q, v, traj, contact, f64(N_DEV, 12), f64(N_DEV, 4), torch.empty(N_DEV, dtype=torch.int32, device="cuda:0")]
    staged = []
    for a in rows(base, N_STAGED):
        b = capi.pinned_empty(a.shape, a.dtype)
        b[:] = a
        staged.append(b)
    d["staged"] = staged + [capi.pinned_empty((N_STAGED, 12)), capi.pinned_empty((N_STAGED, 4)), capi.pinned_empty((N_STAGED,), np.int32)]
    pq, pv = rows(base, N_PLAN)[:2]
    plan_bufs = [capi.pinned_empty(pq.shape), capi.pinned_empty(pv.shape), capi.pinned_empty((N_PLAN,)), capi.pinned_empty((N_PLAN, 12)),
                 capi.pinned_empty((N_PLAN, 4)), capi.pinned_empty((N_PLAN,), np.int32)]
    plan_bufs[0][:], plan_bufs[1][:], plan_bufs[2][:] = pq, pv, np.linspace(0.0, 6.0, N_PLAN)
    d["plan_pinned"] = plan_bufs
    q0 = np.tile(Q0, (N_SMALL, 1))
    d["ro0"] = [cuda(q0), cuda(np.zeros((N_SMALL, 18))), cuda(np.linspace(0.0, 2.0, N_SMALL))]
    d["ro"] = [torch.empty_like(x) for x in d["ro0"]] + [f64(N_SMALL, 12), f64(N_SMALL, 4),
                                                         torch.empty(N_SMALL, dtype=torch.int32, device="cuda:0"), f64(N_SMALL)]
    d["stream"] = torch.cuda.Stream(device=0)
    torch.cuda.synchronize()
    return d


def one_cycle(d):
    """Creates a handle, a plan and a multi-device handle, runs every path that grows device scratch, destroys them all."""
    import torch
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200 import planner as pl
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.rollout import plant_step, rollout
    from quadruped_drake_b200.sharding import MultiGpuController
    from quadruped_drake_b200.wire import WireCodec
    ctl = BatchedController("mini_cheetah", device=0)
    s = pl.TrajectorySampler(ctl, [motion_plan(ctl)])
    q, v, traj, contact = rows(d["base"], N_SMALL)
    t = np.linspace(0.0, 6.0, N_SMALL)

    ctl._check(ctl.lib.wbc_step(ctl._h, capi.WBC_CTRL_ID, N_DEV, C.byref(ctl.make_io(*d["dev"])), None), "wbc_step")
    ctl.step("id", *rows(d["base"], N_PAGEABLE))
    io = capi.WbcIO(*(capi.np_ptr(a) for a in d["staged"]))
    ctl._check(ctl.lib.wbc_step_host(ctl._h, capi.WBC_CTRL_ID, N_STAGED, C.byref(io)), "wbc_step_host")
    hq, hv, ht, htau, hmet, hst = d["plan_pinned"]
    ctl.step_plan("id", s, hq, hv, ht, None, htau, hmet, hst)
    ctl.step_plan("id", s, *rows(d["base"], N_PLAN)[:2], np.linspace(0.0, 6.0, N_PLAN))

    st = d["stream"]
    with torch.cuda.stream(st):
        for x, x0 in zip(d["ro"], d["ro0"]):
            x.copy_(x0)
    rq, rv, rt, rtau, rmet, rso, rerr = d["ro"]
    p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
    rio = capi.WbcRolloutIO(p(rq), p(rv), p(rt), None, p(rtau), p(rmet), p(rso), p(rerr), None)
    ro = capi.WbcRolloutOpts(1, 0, capi.WbcPlantOpts(1.0, 0.2, 30, 0), None)
    ctl._check(ctl.lib.wbc_rollout_ex(ctl._h, capi.WBC_CTRL_ID, s._p, N_SMALL, 3, 5e-3, C.byref(rio), C.byref(ro),
                                      C.c_void_p(st.cuda_stream)), "wbc_rollout_ex")
    st.synchronize()

    ctl.dynamics(q, v)
    ctl.coriolis(q, v)
    codec = WireCodec(ctl)
    codec.decode_trunk_state(codec.encode_trunk_state(t, np.zeros(N_SMALL), traj, contact))
    msgs, _ = codec.encode_robot_state(q, v, np.zeros((N_SMALL, 12)))
    codec.decode_robot_state(msgs)
    s.sample(t, forces=True)
    plant_step(ctl, q, v, np.zeros((N_SMALL, 12)))
    rollout(ctl, s, "id", np.tile(Q0, (N_SMALL, 1)), np.zeros((N_SMALL, 18)), t / 3.0, 3, log_metrics=True)
    rollout(ctl, s, "pd", np.tile(Q0, (N_SMALL, 1)), np.zeros((N_SMALL, 18)), t / 3.0, 3, plant=True)

    m = MultiGpuController("mini_cheetah", devices=[0])
    m.step("id", q, v, traj, contact)
    m.close()
    ctl.close()
    s.close()                      # after its handle
    torch.cuda.synchronize()


def test_second_cycle_leaves_device_memory_where_the_first_left_it(inputs):
    if process_device_bytes() is None:
        pytest.skip("NVML does not list this process (separate PID namespace)")
    one_cycle(inputs)
    first = process_device_bytes()
    one_cycle(inputs)
    second = process_device_bytes()
    assert second == first, f"device memory of the process after the first cycle {first} B, after the second {second} B"
