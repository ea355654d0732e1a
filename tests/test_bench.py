"""bench.py --dump-outputs: the outputs of the last timed step, on inputs that are the same from run to run."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import bench

ROOT = Path(__file__).resolve().parents[1]
DUMPED = ("rows", "tau", "metrics", "status", "qp_info")


def test_dump_rows_whole_batch_or_fixed_sample():
    assert np.array_equal(bench.dump_rows(4096), np.arange(4096))
    big = bench.dump_rows(10**7)
    assert len(big) == bench.DUMP_MAX_ROWS and np.array_equal(big, bench.dump_rows(10**7))
    assert (np.diff(big) > 0).all() and big[0] >= 0 and big[-1] < 10**7
    assert bench.DUMP_MAX_ROWS * 8 * (1 + 12 + 4 + 1 + 4) <= 64 << 20


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"],
                                  ["--workload", "wire", "--dump-outputs", "x"]])
def test_bench_rejects_arguments(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2


@pytest.mark.gpu
def test_dump_outputs_match_library_step(built, tmp_path):
    """Two runs with different step counts dump the same arrays, and they are what the library returns for the same
    seeded batch."""
    import ctypes as C
    import torch
    from quadruped_drake_b200 import capi
    from quadruped_drake_b200.controller import BatchedController
    from quadruped_drake_b200.synth import generate
    n = 1000
    dumps = []
    for steps in (2, 7):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                            "--batch", str(n), "--no-cpu", "--no-e2e", "--no-aux", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        assert sorted(p.name for p in d.iterdir()) == sorted(f"{k}.npy" for k in DUMPED)
        dumps.append({k: np.load(d / f"{k}.npy") for k in DUMPED})
    for k in DUMPED:
        assert dumps[0][k].dtype == np.float64 and np.array_equal(dumps[0][k], dumps[1][k]), k
    assert np.array_equal(dumps[0]["rows"], np.arange(n))

    ctl = BatchedController(bench.ROBOT, device=0)
    try:
        dev = torch.device("cuda:0")
        q, v, traj, contact = generate(ctl.model, n, bench.SEED, bench.PATTERN, ctl.fk)
        tq, tv, tt, tc = (torch.from_numpy(x).to(dev) for x in (q, v, traj, contact))
        tau, met, qi = (torch.empty((n, w), dtype=torch.float64, device=dev) for w in (12, 4, 4))
        st = torch.empty((n,), dtype=torch.int32, device=dev)
        io = ctl.make_io(tq, tv, tt, tc, tau, met, st, None, None, qi)
        stream = torch.cuda.current_stream(dev)
        assert ctl.lib.wbc_step(ctl._h, capi.WBC_CTRL_ID, n, C.byref(io), C.c_void_p(stream.cuda_stream)) == 0
        torch.cuda.synchronize()
    finally:
        ctl.close()
    for k, t in (("tau", tau), ("metrics", met), ("status", st), ("qp_info", qi)):
        assert np.array_equal(dumps[0][k], t.cpu().numpy().astype(np.float64)), k
