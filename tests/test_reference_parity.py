"""Parity with the original ShallowSpeed project: instruction streams of every schedule it implements and the
model partitioner, compared with what its own code produced (``tests/golden/reference_schedules.json``, written
by ``oracle/make_golden.py``)."""
import json
import os

import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_schedules.json")


@pytest.fixture(scope="module")
def ref():
    with open(GOLDEN) as f:
        return json.load(f)


def _stream(sched):
    # same encoding as oracle/make_golden.py: one string per tick, ``Name`` or ``Name:mubatch_id``
    return [" ".join(type(i).__name__ + (f":{i.mubatch_id}" if hasattr(i, "mubatch_id") else "") for i in tick)
            for tick in sched.steps()]


@pytest.mark.parametrize("M", [1, 2, 4, 7])
@pytest.mark.parametrize("S", [1, 2, 4, 8])
def test_instruction_streams_equal_the_reference(ref, M, S):
    from shallowspeed_b200 import pipe

    for ours in (pipe.NaiveParallelSchedule, pipe.GPipeSchedule, pipe.InferenceSchedule):
        for stage in range(S):
            assert _stream(ours(M, S, stage)) == ref["streams"][f"{ours.__name__}/{M}/{S}/{stage}"], (ours.__name__, M, S, stage)


def test_reference_pipedream_is_a_stub_ours_is_not(ref):
    from shallowspeed_b200 import pipe
    from shallowspeed_b200.parallel.validate import validate

    assert ref["pipedream_constructor_raises"] == "NotImplementedError"
    validate(pipe.PipeDreamSchedule, 8, 4)


@pytest.mark.parametrize("pp", [1, 2, 4, 8])
def test_partitioner_matches_reference(ref, pp):
    from shallowspeed_b200.layers import MLP

    sizes = [784, 128, 127, 126, 125, 124, 123, 10]
    assert ref["sizes"] == sizes
    for stage in range(pp):
        r = ref["partition"][f"{pp}/{stage}"]
        o = MLP(sizes, stage, pp, 128)
        assert (o.in_dim, o.out_dim) == (r["in_dim"], r["out_dim"])
        assert [type(l).__name__ for l in o.layers] == r["layers"]
        linears = [l for l in o.layers if type(l).__name__ == "Linear"]
        assert len(linears) == len(r["linears"])
        for lo, lr in zip(linears, r["linears"]):
            assert (lo.activation is not None) == lr["activation"]
            assert list(lo._params["W"].data.shape) == lr["W"]
            assert list(lo._params["b"].data.shape) == lr["b"]
