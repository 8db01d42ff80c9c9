#!/usr/bin/env python
"""Regenerate the reference-parity fixtures under ``tests/golden/`` from a checkout of the original
ShallowSpeed project (NumPy + mpi4py; driven here through ``baseline/mpi_shim``).

    python oracle/make_golden.py [--reference PATH/TO/ShallowSpeed]     # default: the install in oracle/_ref

The tests never import the original project: they compare against what this script stored.

* ``reference_schedules.json``  - instruction streams of NaiveParallel / GPipe / Inference schedules for every
                                 (micro-batches, stages, stage) the tests cover, whether PipeDreamSchedule is
                                 constructible, and the model partition (per stage: dims, layer types,
                                 activations, parameter shapes) of the default MLP for pp = 1, 2, 4, 8.
* ``reference_mlp_numerics.npz`` - the default MLP (784-128-127-126-125-124-123-10, one stage, batch 128):
                                 initial parameters, forward output and gradients of one micro-batch of 32 rows
                                 (inputs: ``np.random.RandomState(0)``).  The output, biases and bias gradients
                                 are stored in full; weights as every row / column sum plus a fixed sample of
                                 elements (``SAMPLE`` seeded flat indices per matrix, stored as ``W<i>_idx``), which
                                 pins down the reference's init recipe.  Every weight gradient is stored as the
                                 two factors the reference multiplies, ``dW<i> = G<i>.T @ A<i>`` (``G<i>``: the layer's output
                                 gradient after the activation's backward, ``A<i>``: its input; ``A0`` is the
                                 regenerable input batch and is not stored), so a test can rebuild it in full.
"""
import argparse
import contextlib
import io
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [784, 128, 127, 126, 125, 124, 123, 10]
MUBATCHES = [1, 2, 4, 7]
STAGES = [1, 2, 4, 8]
SAMPLE = 512


def sample_index(numel: int, i: int) -> np.ndarray:
    """Seeded flat indices into weight matrix ``i`` (stored next to the values)."""
    return np.sort(np.random.RandomState(1000 + i).choice(numel, size=min(numel, SAMPLE), replace=False)).astype(np.int32)


def stream(sched):
    """One string per tick: the tick's instructions as ``Name`` or ``Name:mubatch_id``, space-separated."""
    return [" ".join(type(ins).__name__ + (f":{ins.mubatch_id}" if hasattr(ins, "mubatch_id") else "") for ins in tick)
            for tick in sched.steps()]


def schedules_and_partition(rpipe, rlayers):
    streams = {}
    for cls in (rpipe.NaiveParallelSchedule, rpipe.GPipeSchedule, rpipe.InferenceSchedule):
        for m in MUBATCHES:
            for s in STAGES:
                for stage in range(s):
                    streams[f"{cls.__name__}/{m}/{s}/{stage}"] = stream(cls(m, s, stage))
    try:
        rpipe.PipeDreamSchedule()
        pipedream = None
    except Exception as exc:  # noqa: BLE001 - the exception type is the recorded fact
        pipedream = type(exc).__name__
    partition = {}
    for pp in STAGES:
        for stage in range(pp):
            with contextlib.redirect_stdout(io.StringIO()):
                r = rlayers.MLP(SIZES, stage, pp, 128)
            partition[f"{pp}/{stage}"] = {
                "in_dim": r.in_dim, "out_dim": r.out_dim,
                "layers": [type(layer).__name__ for layer in r.layers],
                "linears": [{"activation": layer.activation is not None, "W": list(layer._params["W"].data.shape),
                             "b": list(layer._params["b"].data.shape)}
                            for layer in r.layers if type(layer).__name__ == "Linear"],
            }
    return {"sizes": SIZES, "streams": streams, "pipedream_constructor_raises": pipedream, "partition": partition}


def mlp_numerics(rlayers):
    with contextlib.redirect_stdout(io.StringIO()):
        ref = rlayers.MLP(SIZES, 0, 1, 128)
    rs = np.random.RandomState(0)
    x = rs.randn(32, 784).astype(np.float32)
    t = np.eye(10, dtype=np.float32)[rs.randint(0, 10, 32)]
    out = ref.forward(x, 0)
    factors = []                           # (G, A) of every Linear's backward, last layer first
    linear_grad = rlayers.linear_grad

    def recording_linear_grad(grad_output, input, weight):
        factors.append((grad_output, input))
        return linear_grad(grad_output, input, weight)

    rlayers.linear_grad = recording_linear_grad
    try:
        ref.backward(t, 0)
    finally:
        rlayers.linear_grad = linear_grad
    factors.reverse()
    arrays = {"out": np.asarray(out, dtype=np.float64)}
    for i, (w, b) in enumerate(zip(ref.parameters()[0::2], ref.parameters()[1::2])):
        # under NumPy >= 2 the reference keeps its weights in fp64; its intended dtype is fp32
        wd, wg = w.data.astype(np.float32), np.asarray(w.grad, dtype=np.float64)
        idx = arrays[f"W{i}_idx"] = sample_index(wd.size, i)
        arrays[f"W{i}_sample"] = wd.reshape(-1)[idx]
        arrays[f"W{i}_rowsum"] = wd.astype(np.float64).sum(axis=1)
        arrays[f"W{i}_colsum"] = wd.astype(np.float64).sum(axis=0)
        arrays[f"b{i}"] = b.data.astype(np.float32)
        arrays[f"db{i}"] = np.asarray(b.grad, dtype=np.float64)
        g, a = (np.asarray(v, dtype=np.float32) for v in factors[i])
        arrays[f"G{i}"] = g
        if i:
            arrays[f"A{i}"] = a
        else:
            assert np.array_equal(a, x)
        rebuilt = g.astype(np.float64).T @ a.astype(np.float64)
        assert np.abs(rebuilt - wg).max() < 1e-9, "stored factors do not rebuild the reference's weight gradient"
    return arrays


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reference", default=os.path.join(ROOT, "oracle", "_ref"),
                    help="checkout of the original ShallowSpeed project (default: what build() installed in oracle/_ref)")
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    args = ap.parse_args()

    sys.path.insert(0, os.path.join(ROOT, "baseline", "mpi_shim"))
    sys.path.insert(0, os.path.abspath(args.reference))
    import shallowspeed.layers as rlayers
    import shallowspeed.pipe as rpipe

    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "reference_schedules.json"), "w") as f:
        json.dump(schedules_and_partition(rpipe, rlayers), f, indent=1)
        f.write("\n")
    np.savez_compressed(os.path.join(args.out, "reference_mlp_numerics.npz"), **mlp_numerics(rlayers))
    print("wrote", sorted(os.listdir(args.out)))


if __name__ == "__main__":
    main()
