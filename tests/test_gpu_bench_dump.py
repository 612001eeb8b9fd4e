"""-m gpu: bench.py --dump-outputs writes the results of the last timed step, row for row the oracle's forward of the
requests that step routed here, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import models

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_holds_the_last_timed_steps_results(tmp_path):
    import torch
    dims, tick, models_per_gpu, W, K = [64, 96, 48, 32], 32, 6, 1, 3
    out = tmp_path / "dump"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", str(W),
                          "--tick", str(tick), "--models-per-gpu", str(models_per_gpu), "--dims", *map(str, dims),
                          "--arena-gib", "1", "--host-gib", "1", "--preheat-s", "0", "--samplers", "none",
                          "--skip-e2e", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert run.returncode == 0, run.stderr[-3000:]
    assert json.loads(run.stdout.strip().splitlines()[-1])["steps"] == K
    y = np.load(out / "predict_y.npy")
    # the last timed step as bench.py plans it (its trace spans warm-up, timed, e2e warm-up and e2e steps)
    wl = bench.build_workload(1, models_per_gpu, tick, W + K + W + K)
    row_models = [m for m, n_local, fl in bench.step_plan(wl, 0, W + K - 1, tick) for _ in range(n_local + len(fl))]
    assert y.dtype == np.float32 and y.shape == (tick, dims[-1]) and len(row_models) == tick
    x = torch.randn(tick * 4, dims[0], device="cuda", dtype=torch.float32,
                    generator=torch.Generator(device="cuda").manual_seed(0)).cpu().numpy()
    for m in set(row_models):
        rows = [i for i, mm in enumerate(row_models) if mm == m]
        man, blob = models.synth_mlp_blob(dims, seed=1000 + m)
        assert np.max(np.abs(y[rows] - models.forward(man, blob, x[rows], np.float64))) <= 1e-4, f"model m{m}"
