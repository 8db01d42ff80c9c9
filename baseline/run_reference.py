"""Run the UNMODIFIED reference (siboehm/ShallowSpeed, installed in oracle/_ref by build()) through
its own public API - the same objects and loop as its train.py:98-146 (MLP, SGD, Dataset,
Worker, schedules) - on MNIST-shaped synthetic data, and time K training steps.

The only things outside the reference's code are (a) the mpi4py shim (no MPI offline),
(b) the data files (synthetic, written in the reference's own on-disk format) and (c) an
fp32 cast of the freshly initialised weights, which restores the reference's intended
NumPy<2 dtype behaviour (SURVEY.md fact 5) - without it the reference silently computes in
fp64 and is ~1.6x slower, so the cast favours the reference.
"""
import argparse
import contextlib
import io
import os
import sys
import time
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF = HERE.parent / "oracle" / "_ref"


def reference_available():
    return (REF / "shallowspeed" / "pipe.py").exists()


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--dp", type=int, default=1)
    ap.add_argument("--pp", type=int, default=1)
    ap.add_argument("--schedule", default="naive", choices=["naive", "gpipe"])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--global-batch-size", type=int, default=128)
    ap.add_argument("--n-mubatches", type=int, default=4)
    ap.add_argument("--data-dir", default="/tmp/ssb_ref_data/mnist_784")
    ap.add_argument("--keep-fp64", action="store_true", help="do not cast the weights back to fp32")
    ap.add_argument("--threads", type=int, default=0,
                    help="BLAS threads per rank; 0 = calibrate: time a few steps at 1,2,4,...,cores/ranks threads and keep the fastest")
    args = ap.parse_args(argv)

    world = args.dp * args.pp
    max_threads = max(1, (os.cpu_count() or 1) // world)
    threads = min(args.threads, max_threads) if args.threads else max_threads
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = str(threads)          # upper bound of the BLAS pool; the sweep below lowers it at run time
    sys.path.insert(0, str(HERE / "mpi_shim"))
    sys.path.insert(0, str(REF))
    import numpy as np
    from mpi4py import MPI
    from shallowspeed.dataset import Dataset
    from shallowspeed.layers import MLP
    from shallowspeed.optimizer import SGD
    from shallowspeed.pipe import GPipeSchedule, NaiveParallelSchedule, Worker
    from shallowspeed.utils import assert_sync, get_model_hash

    assert MPI.COMM_WORLD.size == world, f"world {MPI.COMM_WORLD.size} != dp*pp {world}"
    rank = MPI.COMM_WORLD.Get_rank()
    dp_comm = MPI.COMM_WORLD.Split(color=rank % args.pp)
    pp_comm = MPI.COMM_WORLD.Split(color=rank // args.pp)
    gbs = args.global_batch_size
    layer_sizes = [784, 128, 127, 126, 125, 124, 123, 10]
    with contextlib.redirect_stdout(io.StringIO()):
        model = MLP(layer_sizes, stage_idx=pp_comm.rank, n_stages=args.pp, batch_size=gbs)
    model.train()
    if not args.keep_fp64:
        for p in model.parameters():
            p.data = p.data.astype(np.float32)
    optimizer = SGD(model.parameters(), lr=0.006)
    local_bs = gbs // args.dp
    dataset = Dataset(Path(args.data_dir), global_batch_size=gbs, mubatch_size=local_bs // args.n_mubatches, validation=False)
    dataset.load(dp_comm.Get_rank(), dp_comm.Get_size())
    worker = Worker(dp_comm, pp_comm, model, dataset, optimizer)
    cls = {"naive": NaiveParallelSchedule, "gpipe": GPipeSchedule}[args.schedule]
    n_batches = dataset.get_num_batches()

    def step(i):
        sched = cls(num_micro_batches=args.n_mubatches, num_stages=args.pp, stage_id=pp_comm.rank)
        worker.execute(sched, i % n_batches)

    for i in range(args.warmup):
        step(i)

    # BLAS thread count: 32x784x128 GEMMs are SLOWER on 128 threads than on a few.  The reference sets nothing, so we
    # give it its best case: a short calibration over powers of two (every rank takes the same decision: the times are
    # summed over ranks), then the timed run at the winner.  Outside the reference's code, like the timing itself.
    sweep = None
    if not args.threads:
        try:
            from threadpoolctl import threadpool_limits

            cands = [t for t in (1, 2, 4, 8, 16, 32, 64, 128, 256) if t <= max_threads] or [1]
            cal_steps = 8
            sweep = {}
            for t in cands * 2:                 # two passes, keep the better one per candidate (shared hosts are noisy)
                with threadpool_limits(limits=t):
                    step(0)
                    MPI.COMM_WORLD.Barrier()
                    c0 = time.perf_counter()
                    for i in range(cal_steps):
                        step(i)
                    MPI.COMM_WORLD.Barrier()
                    dt_c = np.array([time.perf_counter() - c0], dtype=np.float64)
                MPI.COMM_WORLD.Allreduce(MPI.IN_PLACE, dt_c, op=MPI.SUM)
                ms = round(1e3 * float(dt_c[0]) / world / cal_steps, 4)
                sweep[t] = min(ms, sweep.get(t, ms))
            threads = min(sweep, key=sweep.get)
            limiter = threadpool_limits(limits=threads)   # stays in force for the timed run
        except ImportError:
            pass
    MPI.COMM_WORLD.Barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    MPI.COMM_WORLD.Barrier()
    dt = time.perf_counter() - t0
    times = MPI.COMM_WORLD.gather(dt, root=0)
    assert_sync(dp_comm, get_model_hash(model))
    if rank == 0:
        dt = max(times)
        return {"ms_per_step": 1e3 * dt / args.steps, "samples_per_s": args.steps * gbs / dt, "threads_per_rank": threads,
                "thread_sweep": sweep,
                "weights_dtype": str(model.parameters()[0].data.dtype)}
    return None


if __name__ == "__main__":
    r = main()
    if r is not None:
        import json

        print(json.dumps(r))
