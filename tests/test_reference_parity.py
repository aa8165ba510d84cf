"""The original ``dfno`` package against this framework's portable backend, from the same weights.

``tests/golden/reference_parity.npz`` holds what the original computed (float64, CPU, gloo) on 1, 2 and 4
ranks -- ``(1,1,2,2,1,1)`` is its in-module demo grid: per rank the state-dict keys and shard shapes, the
distribution info, the output, the relative-L2 loss and the parameter gradients.  Weights, input and target
are seeded draws both sides repeat.  Checked: identical keys and shapes, and outputs, loss and gradients
within 1e-12.

The original imports DistDL and mpi4py; the golden file was made with ``baseline/compat`` standing in for
them.  To regenerate it: ``python tests/test_reference_parity.py --reference-dir DIR``, where ``DIR`` holds
the original ``dfno`` package."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from dfno_b200.utils.testing import run_distributed  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_parity.npz")
CFG = dict(in_shape=[1, 2, 8, 8, 8, 2], nt=4, width=3, modes=(2, 2, 2, 2), blocks=2)
GRIDS = [(1, (1, 1, 1, 1, 1, 1)), (4, (1, 1, 2, 2, 1, 1)), (2, (1, 1, 1, 2, 1, 1))]


def _seeded_state_(net, rank):
    """Fill every floating-point entry of ``net``'s state dict, in sorted key order, from one seeded generator
    (float64 / complex128 draws, so that a float32 buffer on one side does not shift the stream): the same keys
    and shapes give the same weights on both sides."""
    g = torch.Generator().manual_seed(1000 + rank)
    sd = net.state_dict()
    for k, v in sorted(sd.items()):
        if (v.is_floating_point() or v.is_complex()) and v.numel():
            draw = torch.rand(v.shape, dtype=torch.complex128 if v.is_complex() else torch.float64, generator=g)
            sd[k] = ((draw - 0.5) / max(1, v.shape[-1])).to(v.dtype)
    net.load_state_dict(sd)


def _flat_grads(net):
    grads = sorted((k, p.grad) for k, p in net.named_parameters() if p.grad is not None)
    flat = [torch.view_as_real(g).flatten() if g.is_complex() else g.flatten() for _, g in grads]
    return [k for k, _ in grads], torch.cat(flat) if flat else torch.zeros(0, dtype=torch.float64)


def _record(rank, dfno, grid, in_shape, nt, width, modes, blocks, **kw):
    """One rank of a model run with the package ``dfno`` (the original or this framework), ``kw`` to its model."""
    _, P, _ = dfno.create_standard_partitions(grid)
    net = dfno.DistributedFNO(P, in_shape, nt, width, modes, num_blocks=blocks, dtype=torch.float64, **kw)
    _seeded_state_(net, rank)
    info = dfno.compute_distribution_info(P, in_shape)
    x = torch.randn(*in_shape, dtype=torch.float64, generator=torch.Generator().manual_seed(99))
    y = net(x[tuple(info["slice"])].contiguous())
    t = torch.randn(y.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(5 + rank))
    loss = dfno.DistributedRelativeLpLoss(P)(y, t)
    loss.backward()
    grad_keys, grad = _flat_grads(net)
    sd = net.state_dict()
    return {"sd_keys": np.array(sorted(sd)), "sd_shapes": np.array([",".join(map(str, sd[k].shape)) for k in sorted(sd)]),
            "info": np.array([[int(s) for s in info["shape"]], [int(s) for s in info["start"]]]),
            "y": y.detach().numpy(), "loss": np.array(float(loss)), "grad_keys": np.array(grad_keys),
            "grad": grad.numpy()}


def _parity(rank, ws, grid, cfg):
    import warnings
    warnings.filterwarnings("ignore")
    import dfno_b200
    want = np.load(GOLDEN)
    want = {k.split(":", 2)[2]: want[k] for k in want.files if k.startswith(f"ws{ws}:r{rank}:")}
    got = _record(rank, dfno_b200, grid, **cfg, backend="torch", plan="reference")
    assert list(got["sd_keys"]) == list(want["sd_keys"]), "state-dict keys differ"
    assert list(got["sd_shapes"]) == list(want["sd_shapes"]), "state-dict shapes differ"
    assert np.array_equal(got["info"], want["info"]), (got["info"], want["info"])
    assert list(got["grad_keys"]) == list(want["grad_keys"]), "parameters with gradients differ"
    assert got["y"].shape == want["y"].shape and got["grad"].shape == want["grad"].shape
    # off the root the original's loss is mean(empty / empty) = NaN (it only ever prints the root's value);
    # ours is a well-defined 0 there
    lerr = abs(float(want["loss"]) - float(got["loss"])) if rank == 0 else float(got["loss"])
    gerr = float(np.abs(got["grad"] - want["grad"]).max()) if got["grad"].size else 0.0
    return float(np.abs(got["y"] - want["y"]).max()), lerr, gerr


@pytest.mark.parametrize("ws,grid", GRIDS)
def test_unmodified_reference_matches_portable_backend(ws, grid):
    res = run_distributed(_parity, ws, grid, CFG, timeout=600)
    for yerr, lerr, gerr in res:
        assert yerr < 1e-12 and lerr < 1e-12 and gerr < 1e-12, (yerr, lerr, gerr)


def _record_original(rank, ws, ref_dir, grid, cfg):
    import warnings
    warnings.filterwarnings("ignore")
    sys.path[:0] = [os.path.join(ROOT, "baseline", "compat"), ref_dir]
    sys.modules.pop("dfno", None)
    import dfno
    assert os.path.abspath(dfno.__file__).startswith(ref_dir), dfno.__file__
    return _record(rank, dfno, grid, **cfg)


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser(description="regenerate " + os.path.relpath(GOLDEN, ROOT))
    ap.add_argument("--reference-dir", required=True, help="directory that holds the original dfno package")
    ref_dir = os.path.abspath(ap.parse_args().reference_dir)
    arrays = {}
    for ws, grid in GRIDS:
        for rank, rec in enumerate(run_distributed(_record_original, ws, ref_dir, grid, CFG, timeout=600)):
            arrays.update({f"ws{ws}:r{rank}:{k}": v for k, v in rec.items()})
    os.makedirs(os.path.dirname(GOLDEN), exist_ok=True)
    np.savez_compressed(GOLDEN, **arrays)
    print(f"{GOLDEN}: {len(arrays)} arrays, {os.path.getsize(GOLDEN)} bytes")
