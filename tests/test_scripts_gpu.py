"""The reference's two training scripts on a B200: both must run on the fused sm_100a engine (VERDICT r1:
the Navier-Stokes trainer is 2-D + time, the two-phase default config has T = 30), train, checkpoint, resume and
-- for the Navier-Stokes script -- draw its curves / GIF."""
import glob
import os
import subprocess
import sys

import pytest
import torch

from dfno_b200.utils.testing import free_port

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(script_args, nproc, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(free_port())] + script_args
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, OMP_NUM_THREADS="1"), capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    return r.stdout + r.stderr


def _nproc(want):
    return max(n for n in (1, 2, 4) if n <= min(want, torch.cuda.device_count()))


def test_navier_stokes_trainer_runs_on_the_fused_engine(tmp_path):
    n = _nproc(4)
    grid = {1: ["1", "1", "1", "1", "1"], 2: ["1", "1", "2", "1", "1"], 4: ["1", "1", "2", "2", "1"]}[n]   # reference default: 2 x 2
    log = _run(["training/navier_stokes/experiment_navier_stokes.py", "--synthetic", "--grid", "64",
                "--partition-shape", *grid, "--num-data", "40", "--train-split", "0.75", "--in-timesteps", "10", "--out-timesteps", "40",
                "--num-epochs", "3", "--batch-size", "10", "--checkpoint-interval", "3", "--generate-visualization",
                "--out-root", str(tmp_path / "ns")], n)
    assert "backend = fused sm_100a engine" in log, log[-2000:]
    losses = [float(l.split("=")[-1]) for l in log.splitlines() if "average train loss" in l]
    assert len(losses) == 3 and losses[-1] < losses[0], losses
    assert len(glob.glob(str(tmp_path / "ns" / "*" / "model_0003_0000.pt"))) == 1
    assert glob.glob(str(tmp_path / "ns" / "*" / "curves_0003.png")) and glob.glob(str(tmp_path / "ns" / "*" / "sample_0003.gif"))


def test_two_phase_trainer_default_shape_runs_on_the_fused_engine(tmp_path):
    """60 x 60 x 64 x 30, width 20, modes (12, 12, 12, 8): the reference's configuration (train_two_phase.py:14-35)
    on up to 4 GPUs; T = 30 is not a multiple of 4 (padded t pitch)."""
    n = _nproc(4)
    out = str(tmp_path / "tp")
    train = ["training/two_phase/train_two_phase.py", "--num-train", "4", "--num-valid", "1", "--checkpoint-interval", "1",
             "--out-dir", out]
    log = _run(train + ["--epochs", "2"], n)
    assert "backend = fused sm_100a engine" in log and "training finished." in log, log[-2000:]
    assert os.path.exists(os.path.join(out, "model_0002_0000.pt"))
    log = _run(train + ["--epochs", "3", "--resume"], n)
    assert "resumed from epoch 2" in log
    log = _run(["training/two_phase/test_two_phase.py", "--sample", "5", "--out-dir", out], n)
    assert "Saved data sample!" in log


def test_bench_dump_outputs_fused(tmp_path):
    """bench.py --dump-outputs on the fused engine: the loss of the last timed step and the canonical parameters."""
    import json
    import numpy as np
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "2", "--warmup", "3", "--grid", "32",
                        "--modes", "4", "4", "4", "10", "--blocks", "2", "--no-e2e", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    rec = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert rec["impl"] == "fused" and rec["steps"] == 2
    got = {p.name: np.load(p) for p in out.glob("*.npy")}
    assert float(got["loss.npy"]) == np.float32(rec["loss"])
    assert sum(p.stat().st_size for p in out.glob("*.npy")) <= 64 * 10 ** 6
    for k in range(2):                  # [i, o, KX, KY, KZ, mt] complex -> trailing (real, imaginary)
        assert got[f"blocks.{k}.spectral.npy"].shape == (20, 20, 8, 8, 8, 10, 2)
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in got.values())
