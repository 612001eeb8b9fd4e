"""bench.py's host-side plan for the forward hop (N > 1): every request of a tick is executed exactly once by its owner,
forwarded rows get collision-free slots in the ingress rank's window, and all ranks derive the same plan without talking."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_step_plan_partitions_the_tick_and_slots_do_not_collide():
    world, tick = 4, 96
    wl = bench.build_workload(world, 6, tick, 3, forward_frac=0.3)
    tg = tick * world
    assert 0.15 < float(np.mean(wl["ingress"] != wl["dest"])) < 0.45
    for step in range(3):
        lo, hi = step * tg, (step + 1) * tg
        total_rows, slots = 0, {}
        for rank in range(world):
            plan = bench.step_plan(wl, rank, step, tg)
            legacy = dict(bench.step_groups(wl, rank, step, tg)[1])
            assert [m for m, _l, _f in plan] == list(legacy)          # same grouping / order as the N = 1 path
            for m, n_local, fl in plan:
                assert n_local + len(fl) == legacy[m]
                total_rows += n_local + len(fl)
                for p, k in fl:
                    assert p != rank and 0 <= k < tick * 2
                    assert (p, k) not in slots, "two owners would write the same window row"
                    slots[(p, k)] = rank
        assert total_rows == tg
        # the number of window rows used per ingress rank == its forwarded requests in the tick
        fw = wl["ingress"][lo:hi] != wl["dest"][lo:hi]
        for p in range(world):
            n_p = int(np.sum(fw & (wl["ingress"][lo:hi] == p)))
            assert sorted(k for (pp, k) in slots if pp == p) == list(range(n_p))


def test_single_gpu_has_no_forwarding():
    wl = bench.build_workload(1, 8, 64, 2, forward_frac=0.25)
    assert np.array_equal(wl["ingress"], wl["dest"]) and wl["forward_frac"] == 0.0
    assert all(not fl for _m, _n, fl in bench.step_plan(wl, 0, 0, 64))


def test_dumped_sample_is_fixed_ordered_and_bounded():
    y = np.arange(1000 * 16, dtype=np.float32).reshape(1000, 16)
    assert bench.sample_rows(y, y.nbytes) is y
    s = bench.sample_rows(y, 100 * y[0].nbytes + 7)
    assert s.shape == (100, 16) and np.array_equal(s, bench.sample_rows(y, 100 * y[0].nbytes + 7))
    assert np.all(np.diff(s[:, 0]) > 0) and np.all(s[:, 0] % 16 == 0)   # whole rows, in their original order


def test_bench_rejects_runs_without_timed_steps(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args()
