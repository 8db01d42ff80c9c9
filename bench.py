#!/usr/bin/env python
"""Headline benchmark: MLP training throughput (samples/s, whole job) on the reference's
default workload - MLP 784-128-127-126-125-124-123-10, 4 micro-batches, SGD lr 0.006
(BASELINE.md section 2) - data parallel over N B200s.

    python bench.py --gpus N --steps K --warmup W [--impl reference]

* ``value``  : device-timed (CUDA events on the engine's stream, barrier + synchronize on
               both sides, MAX over ranks) with every step's inputs copied from a
               device-resident pool larger than L2.
* ``e2e``    : the same K steps through the public ``Trainer.step`` API with each step's
               inputs copied from PINNED HOST memory (H2D) and its loss read back (D2H).
* scaling    : weak - the per-GPU batch stays at the reference's 128 samples (4 x 32 rows),
               global batch = 128 x N.  ``--scaling strong`` keeps the global batch at 128.
* ``--impl reference`` runs the unmodified reference (NumPy on the host CPUs, mpi4py shim)
               on the same config; N ranks = N processes.
* ``--dump-outputs DIR`` writes the loss and the parameters of the last timed step as .npy files, so that two
               builds run with the same arguments (same seeded inputs and initial weights) can be compared.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LAYER_SIZES = [784, 128, 127, 126, 125, 124, 123, 10]
PER_GPU_BATCH = 128
N_MUBATCHES = 4
LR = 0.006


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak")
    ap.add_argument("--schedule", default="naive")
    ap.add_argument("--comm", choices=["fused", "nccl", "nvls"], default="fused")
    ap.add_argument("--pp-transport", choices=["nccl", "peer"], default=None)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the informational single-GPU tf32-mode measurement")
    ap.add_argument("--precision", choices=["fp32", "tf32"], default="fp32",
                    help="fp32 = 3xTF32 tensor-core products (fp32-equivalent, the reference's contract); tf32 = single pass")
    ap.add_argument("--pp", type=int, default=1, help="pipeline stages (dp = gpus / pp)")
    ap.add_argument("--n-mubatches", type=int, default=N_MUBATCHES)
    ap.add_argument("--hidden", type=int, default=None)
    ap.add_argument("--n-layers", type=int, default=None, help="with --hidden: 784 -> hidden x (n-1) -> 10")
    ap.add_argument("--global-batch", type=int, default=None, help="override the global batch size")
    ap.add_argument("--seed-mode", default="shape")
    ap.add_argument("--pool-batches", type=int, default=352, help="distinct batches in the input pool (352 x 401 KB = 141 MB > L2)")
    ap.add_argument("--repeats", type=int, default=5, help="the K-step block is timed this many times; the MEDIAN block is reported")
    ap.add_argument("--no-exposed", action="store_true", help="skip the compute-only twin run that yields comm.exposed_ms_per_step")
    ap.add_argument("--ref-threads", type=int, default=0, help="reference arm: BLAS threads per rank (0 = calibrate over a sweep)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss of the last step and the parameters it left as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def relaunch_under_torchrun(args):
    """`python bench.py --gpus N` without torchrun: re-exec under torch.distributed.run."""
    import subprocess

    port = 29700 + os.getpid() % 200
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
    sys.exit(subprocess.call(cmd))


def global_batch(args):
    if args.global_batch:
        return args.global_batch
    dp = args.gpus // args.pp
    return PER_GPU_BATCH * dp if args.scaling == "weak" else PER_GPU_BATCH


def layer_sizes(args):
    if args.hidden or args.n_layers:
        return [784] + [args.hidden or 128] * ((args.n_layers or 7) - 1) + [10]
    return list(LAYER_SIZES)


# ----------------------------------------------------------------------------------------
def run_reference(args):
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import run_reference as rr

    if not rr.reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "the original project is not installed in oracle/_ref (build() installs it from a checkout: oracle/install_reference.py)"}))
        return
    rank = int(os.environ.get("RANK", "0"))
    gbs = global_batch(args)
    import tempfile

    # generated on the box (10 s) instead of shipping 200 MB of parquet with every snapshot
    data_dir = os.path.join(tempfile.gettempdir(), "ssb_ref_data", "mnist_784")
    if rank == 0:
        from shallowspeed_b200.dataset import write_reference_files

        write_reference_files(data_dir)
    if args.gpus > 1:   # everyone waits for rank 0's files
        sys.path.insert(0, os.path.join(ROOT, "baseline", "mpi_shim"))
        from mpi4py import MPI

        MPI.COMM_WORLD.Barrier()
    dp = args.gpus // args.pp
    sched = args.schedule
    if sched not in ("naive", "gpipe"):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"the reference's PipeDreamSchedule is a stub that raises "
                              f"(shallowspeed/pipe.py:297-299); schedule '{sched}' cannot run on the reference"}))
        return
    res = rr.main(["--dp", str(dp), "--pp", str(args.pp), "--schedule", sched, "--steps", str(args.steps),
                   "--warmup", str(args.warmup), "--global-batch-size", str(gbs), "--n-mubatches", str(args.n_mubatches),
                   "--data-dir", data_dir, "--threads", str(args.ref_threads)])
    if res is not None:
        print(json.dumps({
            "impl": "reference", "metric": "MLP training samples/sec (whole job)", "value": res["samples_per_s"],
            "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic MNIST-shaped (reference file format), random-init weights",
            "e2e": {"value": res["samples_per_s"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "config": {"model": "MLP 784-128-127-126-125-124-123-10", "global_batch": gbs, "n_mubatches": args.n_mubatches,
                       "parallelism": f"dp{dp}" + (f"xpp{args.pp}" if args.pp > 1 else ""), "schedule": sched,
                       "device": "host CPUs (NumPy + mpi4py shim: " + ("single process" if args.gpus == 1 else
                                  "shared-memory data path, gloo bootstrap" if os.environ.get("SSB_REF_SHM", "1") not in ("0", "")
                                  else "gloo over TCP loopback") + ")",
                       "threads_per_rank": res["threads_per_rank"], "thread_sweep_ms_per_step": res.get("thread_sweep"),
                       "weights_dtype": res["weights_dtype"],
                       "timing": "wall clock between barriers, max over ranks (CPU code)"},
        }))


DUMP_BUDGET = 15_000_000   # float32 values (60 MB): the dump stays under 64 MB with the biases and the loss


def dump_outputs(out_dir, trainer, grid, sizes, loss):
    """What a caller of the timed path holds after its last step, as float32 ``.npy`` files: ``loss`` (shape (1,),
    from the last pipeline stage) and, per layer (global index ``i``), ``W<i>`` (out, in) and ``b<i>`` (out,).
    DP replica 0 writes; each pipeline stage writes its own layers.  When all parameters together exceed
    ``DUMP_BUDGET`` values, every weight matrix is written as ``W<i>_sample``: the elements at a fixed set of flat
    indices drawn from a RandomState seeded with ``i``, so two runs with the same arguments sample the same elements."""
    import numpy as np
    import torch

    from shallowspeed_b200.models.mlp import stage_layer_specs

    if grid.replica != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    trainer.synchronize()
    arena = trainer.model.arena
    total = sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:]))
    frac = min(1.0, DUMP_BUDGET / total)
    for bi, (n_in, n_out, _relu, layer) in enumerate(stage_layer_specs(sizes, grid.stage, grid.pp)):
        w = arena.weight_view(bi)
        if frac < 1.0:
            rs = np.random.RandomState(layer)
            flat = torch.from_numpy(np.sort(rs.randint(0, n_out * n_in, int(frac * n_out * n_in)))).to(w.device)
            np.save(os.path.join(out_dir, f"W{layer}_sample.npy"), w[flat // n_in, flat % n_in].float().cpu().numpy())
        else:
            np.save(os.path.join(out_dir, f"W{layer}.npy"), w.float().cpu().numpy())
        np.save(os.path.join(out_dir, f"b{layer}.npy"), arena.bias_view(bi).reshape(-1).float().cpu().numpy())
    if loss is not None:
        np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float32))


# ----------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from shallowspeed_b200.dataset import synthetic_mnist
    from shallowspeed_b200.parallel.comm import ProcessGrid, make_torch_comms
    from shallowspeed_b200.parallel.engine import Trainer
    from shallowspeed_b200.utils.timing import ClockSampler, max_over_ranks

    world = args.gpus
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        grid = ProcessGrid(world // args.pp, args.pp, rank)
        dp_comm, pp_comm = make_torch_comms(grid)
    else:
        grid, dp_comm, pp_comm = ProcessGrid(1, 1, 0), None, None
    dp = world // args.pp

    gbs = global_batch(args)
    local_bs = gbs // dp
    sizes = layer_sizes(args)
    trainer = Trainer(sizes, global_batch_size=gbs, n_mubatches=args.n_mubatches, lr=LR, schedule=args.schedule,
                      dp_comm=dp_comm if dp > 1 else None, pp_comm=pp_comm if args.pp > 1 else None, grid=grid,
                      comm_mode=args.comm, use_graph=not args.no_graph, device=dev, seed_mode=args.seed_mode,
                      precision=args.precision, pp_transport=args.pp_transport)
    eng = trainer.engine

    # input pools: this replica's shard of `pool` distinct global batches
    pool = args.pool_batches
    if len(sizes) > 9 or max(sizes[1:-1] or [0]) > 2048:
        pool = min(pool, 16)                        # big models: the weights alone dwarf L2
    x, y = synthetic_mnist(n=pool * gbs)
    xs = torch.from_numpy(x[grid.replica::dp].copy()).reshape(pool, local_bs, 784)
    ys = torch.from_numpy(y[grid.replica::dp].copy()).reshape(pool, local_bs, 10)
    x_host, y_host = xs.pin_memory(), ys.pin_memory()
    x_dev, y_dev = xs.to(dev), ys.to(dev)
    h2d = x_host[0].numel() * 4 + y_host[0].numel() * 4
    d2h = 4 * args.n_mubatches

    stream = torch.cuda.ExternalStream(eng.main_stream(), device=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    counter = [0]
    sampler = [None]

    def timed_blocks(step_fn, n, repeats, on_stream):
        """`repeats` blocks of exactly `n` steps, each bracketed by barrier + synchronize on both sides and timed with
        CUDA events on the engine's stream.  One UNTIMED step sits between the opening barrier and the start event: the
        host barrier releases the ranks a few hundred microseconds apart, and with 20 steps of ~0.1 ms that skew would
        otherwise land inside the timed region (round 1: `value` 0.228 ms vs 0.122 ms over 300 steps at N=8).  The
        untimed step's cross-replica flags align the DEVICES, the start event is recorded behind it."""
        out = []
        for _ in range(repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            step_fn(counter[0]); counter[0] += 1
            e0.record(on_stream)
            for _i in range(n):
                step_fn(counter[0]); counter[0] += 1
            e1.record(on_stream)
            if sampler[0] is not None:
                sampler[0].sample_now()                # the device is still working through the block: clocks under load
            barrier()
            out.append(e0.elapsed_time(e1))
        return out

    def reduce_blocks(samples):
        per_block = [max_over_ranks(v, dev) for v in samples]      # max over ranks, block by block
        return sorted(per_block)[len(per_block) // 2], per_block

    def dev_step(i):
        j = i % pool
        trainer.step_async(x_dev[j], y_dev[j])

    losses = []

    def e2e_step(i):
        j = i % pool
        # public API: H2D of this step's inputs from pinned host memory + compute + D2H of its loss, every
        # step; the host consumes the loss of the previous step (one-step-lagged readback) so copies,
        # compute and read-back of neighbouring steps overlap
        losses.append(trainer.step_pipelined(x_host[j], y_host[j]))

    for i in range(max(3, args.warmup)):
        dev_step(counter[0]); counter[0] += 1
    with ClockSampler(local_rank, period_ms=5) as clk:
        sampler[0] = clk
        dev_samples = timed_blocks(dev_step, args.steps, args.repeats, stream)
        for i in range(max(3, args.warmup // 4)):
            e2e_step(counter[0]); counter[0] += 1
        e2e_samples = timed_blocks(e2e_step, args.steps, args.repeats, stream)
        losses.append(trainer.flush())
    sampler[0] = None
    if args.dump_outputs:   # now, while the trainer's last step is the last timed e2e step (SSB_COMM_TIMING runs one more)
        dump_outputs(args.dump_outputs, trainer, grid, sizes, losses[-1])
    ms_dev, dev_blocks = reduce_blocks(dev_samples)
    ms_e2e, e2e_blocks = reduce_blocks(e2e_samples)
    clocks = clk.summary()

    # Exposed (non-overlapped) communication per step = step time of this job minus the step time of the SAME per-GPU
    # work with no communication at all (a second engine on every rank: same layers, same local batch, same 1/global
    # batch loss scale, no DP group), both measured the same way.  Pure-DP jobs only; pipeline jobs report the eager
    # SSB_COMM_TIMING accounting instead (stalls of compute streams on communication events).
    comm = None
    if dp > 1 and args.pp == 1 and not args.no_exposed:
        twin = Trainer(sizes, global_batch_size=gbs, local_batch_size=local_bs, n_mubatches=args.n_mubatches, lr=LR,
                       schedule=args.schedule, use_graph=not args.no_graph, device=dev, seed_mode=args.seed_mode,
                       precision=args.precision)
        tstream = torch.cuda.ExternalStream(twin.engine.main_stream(), device=dev)

        def twin_step(i):
            j = i % pool
            twin.step_async(x_dev[j], y_dev[j])

        for i in range(max(3, args.warmup)):
            twin_step(i)
        ms_twin, twin_blocks = reduce_blocks(timed_blocks(twin_step, args.steps, args.repeats, tstream))
        comm = {"exposed_ms_per_step": max(0.0, ms_dev - ms_twin) / args.steps,
                "compute_only_ms_per_step": ms_twin / args.steps,
                "method": "median step time of this job minus median step time of a communication-free twin engine "
                          "(same per-GPU work, same ranks, same timing harness); max over ranks per block"}
        del twin
    if eng.comm_timing_enabled():   # SSB_COMM_TIMING=1: eager walk with timing events around comm ops and comm waits
        barrier()
        dev_step(0)
        exposed_ms, busy_ms = eng.comm_timing()
        comm = {"exposed_ms_per_step": max_over_ranks(exposed_ms, dev), "busy_ms_per_step": max_over_ranks(busy_ms, dev),
                "method": "eager (no CUDA graph) diagnostic run: waits of compute streams on communication events; "
                          "throughput numbers of this run are not bench values"}

    # Informational: the same workload with single-pass TF32 products (`--precision tf32`), single GPU only.  It never
    # replaces the headline (fp32-equivalent) number and can never take the bench down with it.
    alt = None
    if world == 1 and args.precision == "fp32" and not args.no_alt:
        try:
            t2 = Trainer(sizes, global_batch_size=gbs, n_mubatches=args.n_mubatches, lr=LR, schedule=args.schedule,
                         use_graph=not args.no_graph, device=dev, seed_mode=args.seed_mode, precision="tf32")
            s2 = torch.cuda.ExternalStream(t2.engine.main_stream(), device=dev)

            def alt_step(i):
                j = i % pool
                t2.step_async(x_dev[j], y_dev[j])

            for i in range(max(3, args.warmup)):
                alt_step(i)
            ms_alt, _ = reduce_blocks(timed_blocks(alt_step, args.steps, args.repeats, s2))
            alt = {"precision": "tf32 (single-pass tf32 products, fp32 accumulate)", "value": args.steps * gbs / (ms_alt * 1e-3),
                   "unit": "samples/s", "ms_per_step": ms_alt / args.steps, "note": "informational; the headline value is the fp32-equivalent mode"}
        except Exception as exc:   # noqa: BLE001 - informational only
            alt = {"error": str(exc)[:200]}

    if dp > 1:   # replicas must still be bit-identical after the run
        from shallowspeed_b200.utils import assert_sync, get_model_hash

        trainer.synchronize()
        assert_sync(dp_comm, get_model_hash(trainer.model))
    if rank == 0:
        value = args.steps * gbs / (ms_dev * 1e-3)
        e2e = args.steps * gbs / (ms_e2e * 1e-3)
        kps = int(eng.kernels_per_step())
        print(json.dumps({
            "impl": "ours", "metric": "MLP training samples/sec (whole job)", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": ("fp32 (storage + accumulate fp32; products on tcgen05 as 3xTF32 = lo*hi + hi*lo + hi*hi; measured error vs an fp64 "
                      "oracle at K=784: 6.4e-6 with the default chain-kernel instantiation, 8.5e-7 with SSB_CHAIN_ACC=1, "
                      "cuBLAS fp32 2.9e-7 - profiles/precision_r2.md)"
                      if args.precision == "fp32" else "tf32 (fp32 storage + accumulate, single-pass tf32 products)"),
            "data": "synthetic MNIST-shaped, random-init weights",
            "e2e": {"value": e2e, "unit": "samples/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "block_ms": [round(v, 4) for v in e2e_blocks]},
            "timing": {"blocks": args.repeats, "steps_per_block": args.steps, "block_ms": [round(v, 4) for v in dev_blocks],
                       "reported": "median block (max over ranks per block); one untimed aligning step precedes each start event"},
            "gpu_launches": kps * args.steps,
            "clocks": clocks,
            **({"comm": comm} if comm is not None else {}),
            **({"tf32_mode": alt} if alt is not None else {}),
            "config": {"model": "MLP " + "-".join(str(v) for v in (sizes if len(sizes) <= 9 else sizes[:2] + ["..."] + sizes[-2:])),
                       "global_batch": gbs, "per_replica_batch": local_bs,
                       "n_mubatches": args.n_mubatches, "seq_len": None,
                       "parallelism": f"dp{dp}" + (f"xpp{args.pp}" if args.pp > 1 else ""), "schedule": args.schedule,
                       "dp_comm": args.comm if dp > 1 else "none",
                       "pp_transport": (trainer.worker.pp_transport if args.pp > 1 else "none"), "cuda_graph": (not args.no_graph) and not eng.comm_timing_enabled(),
                       "kernels_per_step": kps, "graph_nodes": int(eng.graph_nodes()),
                       "l2": f"inputs cycle through a pool of {pool} distinct batches ({pool * h2d / 1e6:.0f} MB"
                             + (" > 126 MB L2)" if pool * h2d > 126e6 else ")")
                             + f"; weights of this stage: {trainer.model.arena.weights.numel() * 4 / 1e6:.1f} MB"
                             + (" (legitimately L2-resident across steps)" if trainer.model.arena.weights.numel() * 4 < 20e6 else " (larger than L2: streamed from HBM every step)"),
                       "uses_chain_kernel": bool(eng.uses_chain()) if hasattr(eng, "uses_chain") else None,
                       "last_loss": losses[-1] if losses else None},
        }))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.gpus > 1 and "RANK" not in os.environ:
        relaunch_under_torchrun(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
