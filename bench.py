#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): 3-D Navier-Stokes FNO training step, samples/s.

    python bench.py --gpus N --steps K --warmup W [--impl fused|baseline|reference] [--dump-outputs DIR]

Config: global field 128^3 x 20 t, width 20, modes (12,12,12,10), 4 Fourier blocks, batch 1,
input [1,1,128,128,128,1] -> output [1,1,128,128,128,20]; 1 x N y-pencil over N GPUs (strong
scaling: the global problem is fixed).  A step = forward + relative-L2 loss + backward + Adam.
Synthetic fields, random-init weights.

* ``--impl fused``     this framework's sm_100a engine (default)
* ``--impl baseline``  the same algorithm on stock libraries (torch.fft/cuFFT + cuBLAS + NCCL
                       all_to_all/broadcast/reduce): the re-expression BASELINE.md describes
* ``--impl reference`` the UNMODIFIED reference from baseline/_ref through its own API (its DistributedFNO,
                       loss and training loop: fp32, torch.optim.Adam) -- see baseline/reference_arm.py.  DistDL /
                       mpi4py cannot be installed offline, so its imports resolve to baseline/compat, a
                       self-contained torch.distributed (NCCL) stand-in; nothing of dfno_b200 is on that path.

At N > 1 the fused arm also checks itself: the model and the global sample are functions of a seed only, rank 0
re-runs the same steps on ONE GPU after the timed regions and the JSON line carries ``loss`` and ``loss_parity``
(output of the freshly initialised model N ranks vs 1 rank, loss after the last step); exit code 3 on mismatch.

Timing: W warm-up steps, then K steps between CUDA events bracketed by barrier +
synchronize; max over ranks.  The per-step working set (>= 1.7 GB of activations per block)
is far larger than the 126 MB L2, so no explicit flush is needed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fused", choices=["fused", "baseline", "reference"])
    ap.add_argument("--grid", type=int, default=128)
    ap.add_argument("--nt", type=int, default=20)
    ap.add_argument("--width", type=int, default=20)
    ap.add_argument("--modes", type=int, nargs=4, default=[12, 12, 12, 10])
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--in-channels", type=int, default=1)
    ap.add_argument("--tin", type=int, default=1, help="input time steps (BASELINE config 4 partitions the time axis: use 8)")
    ap.add_argument("--partition", type=int, nargs=6, default=None,
                    help="P_x (default 1 1 1 GPUS 1 1); other grids run the other BASELINE configs, e.g. "
                         "--grid 256 --nt 16 --width 32 --modes 12 12 12 8 --in-channels 2 --partition 1 1 2 2 2 1")
    ap.add_argument("--device", default="cuda", choices=["cuda", "cpu"],
                    help="cpu: dry run of the baseline / reference arms on gloo (host-timed; not a benchmark)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-parity", action="store_true",
                    help="skip the N-rank vs 1-rank output / loss comparison that rank 0 runs after the timed regions")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one produced as DIR/<name>.npy: its loss and the "
                         "updated parameters in the canonical (partition-independent) layout; see dump_outputs()")
    return ap.parse_args()


DUMP_LIMIT = 64 * 10 ** 6    # bytes, all files of --dump-outputs together


def dump_outputs(out_dir, arrays):
    """Write ``{name: tensor}`` as ``out_dir/<name>.npy`` so that two builds can be compared output for output.

    float64 stays float64, every other dtype becomes float32; a complex tensor gains a trailing axis of 2 (real,
    imaginary).  All files together stay within ``DUMP_LIMIT``: arrays are written smallest first, each may take an
    equal share of what is left, and one larger than its share is replaced by a sample of that many elements of its
    flattened form, at sorted indices drawn from a generator seeded with 0 -- the same elements for the same
    arguments, run after run."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for name, t in arrays.items():
        t = t.detach().cpu()
        if t.is_complex():
            t = torch.view_as_real(t)
        out[name] = (t.double() if t.dtype == torch.float64 else t.float()).numpy()
    left = DUMP_LIMIT - 4096 * len(out)                  # room for the .npy headers
    for i, (name, a) in enumerate(sorted(out.items(), key=lambda kv: kv[1].nbytes)):
        n = left // (len(out) - i) // a.itemsize
        if a.size > n:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False, shuffle=False))]
        left -= a.nbytes
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampler running during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        if not self.lines:                       # region shorter than one sampling period: one direct query
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10)
                self.lines = [ln.strip() for ln in out.stdout.splitlines() if ln.strip()]
            except Exception:
                pass
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def main():
    args = parse()
    if args.impl == "reference":
        # the unmodified reference through its own API; nothing of dfno_b200 is imported on this path
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import reference_arm
        return reference_arm.run(args, ClockSampler)

    if args.impl == "baseline":
        os.environ["DFNO_P2P_REPARTITION"] = "0"       # stock NCCL all_to_all / broadcast / reduce only
    import numpy as np
    import torch
    import torch.distributed as dist
    import dfno_b200 as d
    from dfno_b200.parallel.decomposition import assemble_slices, shard_bounds
    from dfno_b200.utils.checkpoint import gather_global_state
    from dfno_b200.utils.env import ensure_process_group

    N = args.gpus
    if N > 1:
        if "RANK" not in os.environ:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
        ensure_process_group()
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    assert world == N, f"world size {world} != --gpus {N}"
    local = int(os.environ.get("LOCAL_RANK", 0))
    on_gpu = args.device == "cuda"
    if on_gpu:
        torch.cuda.set_device(local)
    elif args.impl == "fused":
        raise SystemExit("--impl fused needs --device cuda")
    dev = torch.device("cuda", local) if on_gpu else torch.device("cpu")
    cdtype = torch.bfloat16 if on_gpu else torch.float32      # compute dtype of the fused / baseline arms

    G, T = args.grid, args.nt
    in_shape = [args.batch, args.in_channels, G, G, G, args.tin]
    out_shape = [args.batch, 1, G, G, G, T]
    grid = tuple(args.partition) if args.partition else (1, 1, 1, N, 1, 1)
    if int(torch.tensor(grid).prod()) != N:
        raise SystemExit(f"--partition {grid} does not hold --gpus {N} ranks")
    _, P_x, P_0 = d.create_standard_partitions(grid)
    SEED = 1234

    def build(P, backend):
        if backend == "fused":
            net_ = d.DistributedFNO(P, in_shape, T, args.width, args.modes, num_blocks=args.blocks, device=dev,
                                    dtype=torch.bfloat16, backend="fused", init_seed=SEED)
            return net_, d.FusedAdam(net_, lr=1e-3)
        net_ = d.DistributedFNO(P, in_shape, T, args.width, args.modes, num_blocks=args.blocks, device=dev,
                                dtype=cdtype, backend="torch", init_seed=SEED)
        return net_, torch.optim.Adam([p for p in net_.parameters() if p.numel() > 0], lr=1e-3)

    net, opt = build(P_x, "fused" if args.impl == "fused" else "torch")
    in_dtype = torch.float32 if args.impl == "fused" else cdtype
    crit = d.DistributedRelativeLpLoss(P_x, engine=net if args.impl == "fused" else None)

    # the GLOBAL synthetic sample is a function of the seed only (every rank draws it and keeps its shard), so runs
    # at different world sizes see the same data -- the basis of the loss-parity check below
    gen = torch.Generator(device=dev).manual_seed(SEED)
    x_glob = torch.randn(*in_shape, device=dev, generator=gen)
    # target: a smooth function of the input field plus noise, so the loss actually moves during the timed steps
    # (pure noise would pin the relative L2 loss at 1.0 and make the N-rank vs 1-rank loss check vacuous)
    tt = torch.arange(T, device=dev, dtype=torch.float32)
    y_glob = 0.5 * x_glob[:, :1, ..., :1] * torch.cos(0.3 * tt) + 0.1 * torch.randn(*out_shape, device=dev, generator=gen)
    xi, yi = d.compute_distribution_info(P_x, in_shape), d.compute_distribution_info(P_x, out_shape)
    x_host = x_glob[tuple(xi["slice"])].to(in_dtype).contiguous().cpu()
    y_host = y_glob[tuple(yi["slice"])].contiguous().cpu()
    if args.partition:
        args.no_parity = True            # general partitions are run for size (configs 3 / 4): a 1-rank replay would not fit
    keep_global = args.impl == "fused" and N > 1 and rank == 0 and not args.no_parity
    if not keep_global:
        del x_glob, y_glob
    if on_gpu:
        x_host, y_host = x_host.pin_memory(), y_host.pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)

    # ---- N-rank vs 1-rank, part 1: the forward of the freshly initialised model, gathered on rank 0 (compared below)
    parity, out_cat = None, None
    if args.impl == "fused" and N > 1 and not args.no_parity:
        with torch.no_grad():
            out_n = net(x_dev).float().contiguous()
        shards = [torch.empty_like(out_n) for _ in range(N)] if rank == 0 else None
        dist.gather(out_n, shards, dst=0)
        if rank == 0:
            out_cat = torch.empty(*out_shape, device=dev)
            for r, sh in enumerate(shards):                  # world rank r sits at grid index unravel(r, grid)
                lo, hi = shard_bounds(out_shape, grid, [int(v) for v in np.unravel_index(r, grid)])
                out_cat[assemble_slices(lo, hi)] = sh
            parity = {}
        del out_n, shards

    use_graph = args.impl == "fused" and not args.no_graph
    tr = d.Trainer(net, crit, opt, device=dev, cuda_graph=use_graph)
    steps_taken = [0]

    def step_device():
        steps_taken[0] += 1
        return tr.step_on_device(x_dev, y_dev)

    def step_e2e():
        steps_taken[0] += 1
        return tr.step(x_host, y_host, next_batch=(x_host, y_host))

    def sync_all():
        if N > 1:
            dist.barrier()
        if on_gpu:
            torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        if on_gpu:
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
        else:
            import time
            t0 = time.perf_counter()
        last = None
        for _ in range(steps):
            last = fn()
        if on_gpu:
            e.record()
        sync_all()
        elapsed = s.elapsed_time(e) if on_gpu else (time.perf_counter() - t0) * 1e3
        ms = torch.tensor([elapsed], device=dev, dtype=torch.float64)
        if N > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    sampler = ClockSampler(local)
    if rank == 0 and on_gpu:
        sampler.start()                          # covers warm-up + timed region (identical load)
    for _ in range(max(args.warmup, 3)):
        step_device()
    counter = getattr(net, "_C", None)
    c0 = counter.count if hasattr(counter, "count") else 0
    total_ms, last_loss = timed(step_device, args.steps)
    launches = (counter.count - c0) if hasattr(counter, "count") else 0
    clocks = sampler.stop() if rank == 0 else None
    ms_step = total_ms / args.steps
    value = args.batch * 1000.0 / ms_step
    loss_value = float(last_loss)
    if args.dump_outputs:
        state = gather_global_state(net)                     # collective; the canonical state lands on rank 0
        if rank == 0:
            dump_outputs(args.dump_outputs, {"loss": last_loss, **state})

    # ---- end to end through the public Trainer API: pinned host batch in, loss out
    e2e = None
    if not args.no_e2e:
        for _ in range(3):
            step_e2e()
        e2e_ms, last_loss = timed(step_e2e, args.steps)
        loss_value = float(last_loss)
        e2e = {"value": args.batch * 1000.0 / (e2e_ms / args.steps), "unit": "samples/s",
               "ms_per_step": e2e_ms / args.steps, "h2d_bytes_per_step": tr.h2d_bytes, "d2h_bytes_per_step": tr.d2h_bytes,
               "cuda_graph": bool(tr._graph is not None),
               "how": "Trainer.step(): pinned host batch -> async H2D (double buffered) -> fwd+loss+bwd+Adam -> loss D2H"}

    peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30 if on_gpu else None     # before the 1-rank replay below

    # ---- N-rank vs 1-rank, part 2 (not timed; the other ranks wait at the barrier): rank 0 builds the SAME model
    # (same seed) on ONE GPU, compares its initial output with the gathered N-rank one, repeats the same number of
    # optimisation steps on the same global sample and compares the loss after the last step
    if parity is not None:
        P_1 = d.Partition([0], [1] * 6)
        net1, opt1 = build(P_1, "fused")
        with torch.no_grad():
            out_1 = net1(x_glob).float()
        parity["output_rel_err_vs_1rank_initial"] = float((out_cat - out_1).norm() / out_1.norm().clamp_min(1e-30))
        del out_cat, out_1
        crit1 = d.DistributedRelativeLpLoss(P_1)
        x1, y1 = x_glob.to(in_dtype), y_glob
        l1 = None
        for _ in range(steps_taken[0]):
            opt1.zero_grad()
            l1 = crit1(net1(x1), y1)
            l1.backward()
            opt1.step()
        l1 = float(l1.detach())
        parity.update({"steps": steps_taken[0], "loss_n_ranks": loss_value, "loss_1_rank": l1,
                       "abs_diff": abs(loss_value - l1)})
        parity["ok"] = bool(parity["abs_diff"] < 2e-3 * max(1.0, abs(l1)) and
                            parity["output_rel_err_vs_1rank_initial"] < 2e-2)
        if not parity["ok"]:
            print(f"[bench] LOSS PARITY FAILED: {parity}", file=sys.stderr)

    if rank == 0:
        out = {
            "metric": "3D Navier-Stokes FNO training step (fwd+loss+bwd+Adam) samples/sec, whole job, device-timed, max over ranks",
            "value": value, "unit": "samples/s", "n_gpus": N, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16" if on_gpu else "fp32", "data": "synthetic (random input field, target = smooth function of it + noise; random-init weights)", "impl": args.impl,
            "config": {"model": f"FNO3d+t {G}^3x{T}t width {args.width} modes {tuple(args.modes)} blocks {args.blocks}",
                       "global_batch": args.batch, "seq_len": G * G * G * T,
                       "parallelism": (f"y-pencil 1x{N} (model parallel: field over y, spectral weights over kz)"
                                       if not args.partition else f"P_x = {grid} (model parallel domain decomposition)"),
                       "l2": "per-step working set (>=0.2 GB/rank/block activations) exceeds the 126 MB L2; no flush needed",
                       "step": "forward + DistributedRelativeLpLoss + backward + Adam"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "cuda_graph": bool(tr._graph is not None), "loss": loss_value, "loss_parity": parity,
            "peak_mem_gb": peak_mem,
        }
        print(json.dumps(out))
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    return 0 if (parity is None or parity.get("ok", True)) else 3


if __name__ == "__main__":
    sys.exit(main())
