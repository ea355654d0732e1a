"""Launch schedule of the step entry points: the kernels one call issues (wbc_launch_count) on both sides of every size
threshold of the chunking policies in csrc/wbc_api.cu. The parity tests pin the outputs along these paths; a schedule
change leaves every output bit as it is, so it is pinned here. A reduce -> solve chain counts 2, a PD step and a sampler
call 1 each."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
BASE = 4096


@pytest.fixture(scope="module")
def ctl(built):
    from quadruped_drake_b200.controller import BatchedController
    c = BatchedController("mini_cheetah", device=0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def base(ctl):
    from quadruped_drake_b200.synth import generate
    return generate(ctl.model, BASE, 7, "mixed", ctl.fk)


def rows(base, n):
    idx = np.arange(n) % BASE
    return [np.ascontiguousarray(a[idx]) for a in base]


def launches(ctl, call):
    l0 = ctl.launches
    call()
    return ctl.launches - l0


@pytest.mark.parametrize("n,expect", [(4095, 2), (4096, 4), (5119, 4), (5120, 6), (7167, 6), (7168, 8), (65536, 8), (65537, 2),
                                      (262144, 2), (262145, 4)])
def test_device_step(ctl, base, n, expect):
    """wbc_step on device buffers: 2-4 chains from 4096 to 65536 instances, one chain per 262144 instances otherwise."""
    import torch
    t = [torch.from_numpy(a).to("cuda:0") for a in rows(base, n)]
    assert launches(ctl, lambda: ctl.step("id", *t)) == expect
    torch.cuda.synchronize()


def test_profile_step_is_one_chain_per_rep(ctl, base):
    import torch
    from quadruped_drake_b200 import capi
    n, reps = 4096, 5
    q, v, traj, contact = [torch.from_numpy(a).to("cuda:0") for a in rows(base, n)]
    tau = torch.empty((n, 12), dtype=torch.float64, device="cuda:0")
    met = torch.empty((n, 4), dtype=torch.float64, device="cuda:0")
    st = torch.empty((n,), dtype=torch.int32, device="cuda:0")
    io = ctl.make_io(q, v, traj, contact, tau, met, st)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ms_r, ms_s = C.c_double(), C.c_double()
    assert launches(ctl, lambda: ctl._check(ctl.lib.wbc_profile_step(ctl._h, capi.WBC_CTRL_ID, n, C.byref(io), reps, stream,
                                                                     C.byref(ms_r), C.byref(ms_s)), "wbc_profile_step")) == 2 * reps


def step_host(ctl, base, kind, n, pinned):
    """One wbc_step_host call on page-locked (pinned) or pageable buffers; PD passes q, v and tau only."""
    from quadruped_drake_b200 import capi
    alloc = capi.pinned_empty if pinned else (lambda shape, dtype=np.float64: np.empty(shape, dtype))
    bufs = []

    def put(a):
        b = alloc(a.shape, a.dtype)
        b[:] = a
        bufs.append(b)
        return capi.np_ptr(b)
    q, v, traj, contact = rows(base, n)
    tau = put(np.zeros((n, 12)))
    if kind == "pd":
        io = capi.WbcIO(put(q), put(v), None, None, tau, None, None, None, None, None)
    else:
        io = capi.WbcIO(put(q), put(v), put(traj), put(contact), tau, put(np.zeros((n, 4))), put(np.zeros(n, np.int32)),
                        None, None, None)
    k = {"id": capi.WBC_CTRL_ID, "clf": capi.WBC_CTRL_CLF, "pc": capi.WBC_CTRL_PC, "mptc": capi.WBC_CTRL_MPTC, "pd": capi.WBC_CTRL_PD}[kind]
    ctl._check(ctl.lib.wbc_step_host(ctl._h, k, n, C.byref(io)), "wbc_step_host")


@pytest.mark.parametrize("kind,n,expect", [
    # zero-copy: two halves from 4096 instances; inputs through the copy engine from 24576 (PC / MPTC: 131072) instances,
    # in four chunks below 98304 instances and in chunks of n / 8 clamped to [16384, 32768] from there on
    ("id", 4095, 2), ("id", 4096, 4), ("id", 24575, 4), ("id", 24576, 8), ("id", 98303, 8), ("id", 98304, 12),
    ("clf", 24576, 8), ("pc", 4096, 4), ("pc", 24576, 4), ("pc", 131071, 4), ("pc", 131072, 16), ("mptc", 131072, 16),
    # PD: the same chunk counts, one kernel per chunk
    ("pd", 4095, 1), ("pd", 4096, 2), ("pd", 24575, 2), ("pd", 24576, 4)])
def test_step_host_page_locked(ctl, base, kind, n, expect):
    assert launches(ctl, lambda: step_host(ctl, base, kind, n, True)) == expect


@pytest.mark.parametrize("kind,n,expect", [
    # two chunks from 2048 instances, chunks of n / 8 clamped to [8192, 65536] from 32768 on
    ("id", 2047, 2), ("id", 2048, 4), ("id", 32767, 4), ("id", 32768, 8), ("id", 40000, 10), ("id", 131072, 16),
    ("pd", 2047, 1), ("pd", 2048, 2)])
def test_step_host_pageable(ctl, base, kind, n, expect):
    assert launches(ctl, lambda: step_host(ctl, base, kind, n, False)) == expect


@pytest.mark.parametrize("n,pinned,expect", [(4095, True, 3), (4096, True, 5), (4096, False, 3)])
def test_step_plan_host(ctl, base, n, pinned, expect):
    """wbc_step_plan_host: one sampler call, then the step as two halves from 4096 instances on page-locked buffers and as
    one chain on pageable ones."""
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200 import planner as pl
    bh = float(ctl.model.nominal_q()[6])
    s = pl.TrajectorySampler(ctl, [pl.make_motion_plan("mini_cheetah", "standing", 6.0, base_height=bh)])
    q, v, _, _ = rows(base, n)
    t = np.linspace(0.0, 6.0, n)
    alloc = capi.pinned_empty if pinned else (lambda shape, dtype=np.float64: np.empty(shape, dtype))
    hq, hv, ht = alloc((n, 19)), alloc((n, 18)), alloc((n,))
    hq[:], hv[:], ht[:] = q, v, t
    tau, met, st = alloc((n, 12)), alloc((n, 4)), alloc((n,), np.int32)
    assert launches(ctl, lambda: ctl.step_plan("id", s, hq, hv, ht, None, tau, met, st)) == expect
    s.close()
