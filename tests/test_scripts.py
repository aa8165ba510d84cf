"""End-to-end runs of the user-facing scripts on CPU (gloo, 2 ranks, tiny problems): the two
trainers incl. resume + inference, the reference-style benchmark harness + script generator, the
stand-alone gradient-check tool and the in-module demo.  These are what a user of the reference
would launch with mpirun (SURVEY.md C7-C13)."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from dfno_b200.utils.testing import free_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(script_args, nproc=2, timeout=420, cwd=ROOT):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(free_port())] + script_args
    env = dict(os.environ, OMP_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-3000:]
    return r.stdout


@pytest.mark.slow
def test_two_phase_train_resume_infer(tmp_path):
    out = str(tmp_path / "tp")
    common = ["--shape", "8", "8", "8", "4", "--modes", "2", "2", "2", "2", "--width", "4"]
    train = ["training/two_phase/train_two_phase.py", *common, "--num-train", "3", "--num-valid", "2",
             "--checkpoint-interval", "1", "--out-dir", out]
    log = _run(train + ["--epochs", "2"])
    assert "training finished." in log
    for r in (0, 1):
        assert os.path.exists(os.path.join(out, f"model_0002_{r:04d}.pt")) and os.path.exists(os.path.join(out, f"model_{r:04d}.pt"))
    log = _run(train + ["--epochs", "3", "--resume"])
    assert "resumed from epoch 2" in log and os.path.exists(os.path.join(out, "model_0003_0001.pt"))
    hist = json.load(open(os.path.join(out, "loss_epoch_2.json")))
    assert len(hist["train"]) == 3                     # two epochs before the interruption + one after
    recs = [json.loads(l) for l in open(os.path.join(out, "metrics_0000.jsonl"))]
    assert any("valid_loss" in r for r in recs)
    log = _run(["training/two_phase/test_two_phase.py", *common, "--sample", "4", "--out-dir", out])
    assert "Saved data sample!" in log and os.path.exists(os.path.join(out, "fno_sample.npz"))


@pytest.mark.slow
def test_navier_stokes_experiment(tmp_path):
    log = _run(["training/navier_stokes/experiment_navier_stokes.py", "--synthetic", "--grid", "16",
                "--partition-shape", "1", "1", "2", "1", "1", "--num-data", "6", "--in-timesteps", "2",
                "--out-timesteps", "4", "--width", "4", "--modes", "2", "2", "2", "--num-blocks", "1",
                "--num-epochs", "2", "--batch-size", "2", "--checkpoint-interval", "1",
                "--out-root", str(tmp_path / "ns")])
    assert "average test mse" in log
    assert len(glob.glob(str(tmp_path / "ns" / "*" / "model_0002_000[01].pt"))) == 2


def test_reference_style_benchmark_and_generator(tmp_path):
    out = str(tmp_path / "bench")
    for kind in ("eval", "grad"):
        _run(["benchmarks/bench.py", "--input-shape", "1", "1", "8", "8", "8", "1", "--partition_shape", "1", "1", "1", "2", "1", "1",
              "--width", "4", "--modes", "2", "2", "2", "2", "--num-timesteps", "4", "--device", "cpu",
              "--benchmark-type", kind, "--output-dir", out, "--dtype", "fp32"])
    files = sorted(glob.glob(os.path.join(out, "*.json")))
    assert len(files) == 4                             # {eval, grad} x 2 ranks
    rec = json.load(open([f for f in files if "grad" in f][0]))
    assert {"dt", "dt_comm", "dt_comp", "dt_grad"} <= set(rec)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "benchmarks", "gen_scripts.py"), "--system", "local",
                        "--max-workers", "4", "--out", str(tmp_path / "gen")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    names = {os.path.basename(p) for p in glob.glob(str(tmp_path / "gen" / "*.sh"))}
    assert {"eval_weak_scaling_spatial_gpu.sh", "grad_weak_scaling_temporal_gpu.sh", "submit_local.sh"} <= names


def test_gradient_check_tool_cli():
    log = _run(["tools/gradient_check.py", "--case", "transpose-linear"])
    assert "passed gradcheck [transpose-linear]" in log and "failed" not in log


def test_bench_contract_dry_run():
    """bench.py on CPU (host-timed dry run): JSON contract keys, the reference arm's `unavailable`
    line without a GPU, and the reference arm (unmodified reference model code on baseline/compat) on gloo."""
    small = ["--device", "cpu", "--grid", "16", "--nt", "8", "--width", "4", "--modes", "2", "2", "2", "2",
             "--blocks", "1", "--steps", "2", "--warmup", "3"]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT)
    ref = json.loads(r.stdout.strip().splitlines()[-1])
    assert r.returncode == 0 and ref["impl"] == "reference" and ("unavailable" in ref or "value" in ref)
    impls = ["baseline"] + (["reference"] if os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "dfno")) else [])
    for impl in impls:
        out = _run(["bench.py", "--gpus", "2", "--impl", impl, *small])
        rec = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                    "scaling", "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches"):
            assert key in rec, key
        assert rec["n_gpus"] == 2 and rec["steps"] == 2 and rec["warmup"] == 3 and rec["impl"] == impl
        assert "h2d_bytes_per_step" in rec["e2e"] and rec["value"] > 0      # bytes are 0 in the CPU dry run


def test_bench_dump_outputs_dry_run(tmp_path):
    """--dump-outputs: the loss of the last timed step and the updated canonical parameters, the same from run to
    run with the same arguments."""
    small = ["--device", "cpu", "--grid", "16", "--nt", "8", "--width", "4", "--modes", "2", "2", "2", "2",
             "--blocks", "1", "--steps", "2", "--warmup", "3", "--no-e2e"]
    dumps = []
    for i in range(2):
        out = _run(["bench.py", "--gpus", "2", "--impl", "baseline", *small, "--dump-outputs", str(tmp_path / str(i))])
        rec = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
        files = sorted(glob.glob(str(tmp_path / str(i) / "*.npy")))
        dumps.append({os.path.basename(f): np.load(f) for f in files})
        assert sum(os.path.getsize(f) for f in files) <= 64 * 10 ** 6
        assert all(a.dtype in (np.float32, np.float64) for a in dumps[-1].values())
        assert float(dumps[-1]["loss.npy"]) == np.float32(rec["loss"])
        assert dumps[-1]["blocks.0.spectral.npy"].shape[-1] == 2 and "linear1.W.npy" in dumps[-1]
    assert dumps[0].keys() == dumps[1].keys()
    for k in dumps[0]:
        assert np.array_equal(dumps[0][k], dumps[1][k]), k


def test_bench_dump_outputs_samples_within_the_limit(tmp_path, monkeypatch):
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("bench_main", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 1 << 20)
    arrays = {"big": torch.arange(1 << 20, dtype=torch.float32), "w": torch.randn(3, 4, dtype=torch.complex64),
              "loss": torch.tensor(0.5, dtype=torch.float64)}
    for i in range(2):
        bench.dump_outputs(str(tmp_path / str(i)), arrays)
    assert sum(os.path.getsize(f) for f in glob.glob(str(tmp_path / "0" / "*.npy"))) <= 1 << 20
    big = np.load(tmp_path / "0" / "big.npy")
    assert big.ndim == 1 and 0.9 * (1 << 18) < big.size < 1 << 18     # what the small arrays leave of 1 MiB
    assert np.all(np.diff(big) > 0)                                   # distinct elements, in order
    assert np.array_equal(big, np.load(tmp_path / "1" / "big.npy"))
    w = np.load(tmp_path / "0" / "w.npy")
    assert w.dtype == np.float32 and np.array_equal(w, torch.view_as_real(arrays["w"]).numpy())
    loss = np.load(tmp_path / "0" / "loss.npy")
    assert loss.dtype == np.float64 and float(loss) == 0.5
