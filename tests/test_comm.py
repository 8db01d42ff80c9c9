"""Process grid + communicator plumbing (CPU)."""
import threading

import pytest

import torch

from shallowspeed_b200.parallel.comm import ProcessGrid, SelfComm, ThreadFabric


def test_process_grid_matches_reference_rank_mapping():
    # reference train.py:89-92: dp_comm = Split(color = rank % PP), pp_comm = Split(color = rank // PP)
    dp, pp = 2, 4
    for r in range(dp * pp):
        g = ProcessGrid(dp, pp, r)
        assert g.stage == r % pp and g.replica == r // pp
        assert g.dp_group_ranks() == [x for x in range(dp * pp) if x % pp == r % pp]
        assert g.pp_group_ranks() == [x for x in range(dp * pp) if x // pp == r // pp]
        assert g.pp_group_ranks() == list(range(g.replica * pp, g.replica * pp + pp))   # adjacent ranks = adjacent GPUs


def test_self_comm_is_a_noop_communicator():
    c = SelfComm()
    t = torch.ones(4)
    c.iallreduce(t).wait()
    assert torch.equal(t, torch.ones(4)) and c.gather("h") == ["h"] and c.Get_size() == 1 and c.Get_rank() == 0


def test_thread_fabric_allreduce_is_rank_ordered_and_p2p_works():
    n = 4
    fab = ThreadFabric(n)
    out = {}

    def main(rank):
        c = fab.comm(rank)
        t = torch.full((8,), float(rank + 1))
        c.allreduce(t)
        out[rank] = t.clone()
        if rank == 0:
            c.send(torch.arange(3.0), 1)
        if rank == 1:
            buf = torch.empty(3)
            c.recv(buf, 0)
            out["recv"] = buf
        out[("g", rank)] = c.gather(rank * 10)

    th = [threading.Thread(target=main, args=(r,)) for r in range(n)]
    [t.start() for t in th]
    [t.join(30) for t in th]
    for r in range(n):
        assert torch.equal(out[r], torch.full((8,), 10.0))      # 1+2+3+4, identical bits on every rank
    assert torch.equal(out["recv"], torch.arange(3.0))
    assert out[("g", 0)] == [0, 10, 20, 30] and out[("g", 1)] is None


def test_watchdog_reports_and_aborts_on_timeout(monkeypatch):
    """Failure detection (host side): a step that never finishes raises StepTimeout, names the rank and
    aborts the native communicators so peers do not hang with it."""
    from shallowspeed_b200.parallel import engine as E

    monkeypatch.delenv("SSB_WATCHDOG_S", raising=False)
    assert E.watchdog_seconds() is None and E.watchdog_seconds(0) is None and E.watchdog_seconds(2) == 2.0
    monkeypatch.setenv("SSB_WATCHDOG_S", "7.5")
    assert E.watchdog_seconds() == 7.5 and E.watchdog_seconds(1) == 1.0

    class FakeEngine:
        def __init__(self, done):
            self.done, self.waited = done, None

        def wait(self, t):
            self.waited = t
            return self.done

        def comm_status(self):
            return "pp_comm=unhandled cuda error "

        def describe(self):
            return "plan"

    class FakeNccl:
        aborted = False

        def abort(self):
            self.aborted = True

    w = E.NativeWorker.__new__(E.NativeWorker)
    w.stage_id, w.dp_comm, w._pp_nccl, w._dp_nccl = 1, SelfComm(), FakeNccl(), None
    ok = FakeEngine(True)
    w.guard(ok, 3.0)
    assert ok.waited == 3.0 and not w._pp_nccl.aborted
    w.guard(FakeEngine(False), None)            # disabled watchdog never waits
    with pytest.raises(E.StepTimeout, match="stage 1.*unhandled cuda error"):
        w.guard(FakeEngine(False), 0.01, what="step 12")
    assert w._pp_nccl.aborted


def test_fd_passing_over_unix_socket(request):
    """NVLS set-up hands the multicast object's POSIX fd to the other replicas with SCM_RIGHTS; check the transport
    with a pipe: what the peers write into the received descriptors arrives at the leader's read end."""
    import os
    import shutil
    import tempfile

    from shallowspeed_b200.parallel import engine as E

    # AF_UNIX socket paths are limited to 107 bytes, which pytest's tmp_path under a deep $TMPDIR can exceed
    sock_dir = tempfile.mkdtemp(prefix="ssb_fd_", dir="/tmp")
    request.addfinalizer(lambda: shutil.rmtree(sock_dir, ignore_errors=True))
    r, w = os.pipe()
    path = os.path.join(sock_dir, "fd.sock")
    srv = E.serve_fd(path, w, 2)
    got = []

    def peer(i):
        fd = E.recv_fd(path, timeout_s=20)
        os.write(fd, bytes([65 + i]))
        os.close(fd)
        got.append(i)

    ts = [threading.Thread(target=peer, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    E.serve_fd_finish(srv, path, w, 2)
    for t in ts:
        t.join(30)
    os.close(w)
    assert sorted(os.read(r, 16)) == [65, 66] and sorted(got) == [0, 1]
    os.close(r)
    assert not os.path.exists(path)


def test_nvls_requires_support_and_is_reported_unavailable_on_cpu():
    from shallowspeed_b200 import _C

    assert _C.NvlsContext.supported() in (False, True)
    from shallowspeed_b200.parallel.engine import DP_MODE

    assert DP_MODE["nvls"] == 3
