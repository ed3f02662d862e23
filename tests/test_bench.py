"""bench.py --dump-outputs: the files hold F and G of the LAST timed evaluation, i.e. of the hyper-parameters of step
warmup + steps - 1 of the benchmark's trajectory, checked against the CPU oracle at a small N."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import gpr_oracle as o

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_last_timed_step(tmp_path):
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    N, steps, warmup = 2048, 3, 2
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                        "--n", str(N), "--no-cpu", "--no-predict", "--no-sharded", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup
    F, G = np.load(out / "F.npy"), np.load(out / "G.npy")
    assert F.dtype == np.float64 and G.dtype == np.float64 and F.shape == (1,) and G.shape == (19,)
    assert F[0] == line["F_last"]
    x, y, hp0 = bench.make_problem(N, bench.D_FULL)
    hp = bench.hp_at(hp0, warmup + steps - 1)
    Fo, Go = o.log_loss_grad(np.log(hp), o.GPRModel((o.SE, o.SE, o.NOISE), hp, x, y))
    assert abs(F[0] - Fo) <= 1e-8 * abs(Fo), (F[0], Fo)
    assert np.all(np.abs(G - Go) <= 1e-8 * np.maximum(np.abs(Go), 1e-8 * np.linalg.norm(Go))), (G, Go)
