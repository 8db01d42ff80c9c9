"""CLI-level smoke tests on the CPU: train.py (sequential and a spawned DP x PP grid through the
portable VM), checkpoint/resume, and the JSON contract of bench.py's reference arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
    env = dict(os.environ, OMP_NUM_THREADS="2")
    return subprocess.run([sys.executable] + args, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)


def test_train_sequential_cpu(tmp_path):
    log = tmp_path / "m.jsonl"
    r = _run(["train.py", "--device", "cpu", "--steps", "6", "--no-eval", "--synthetic", "--log-json", str(log),
              "--save", str(tmp_path / "ck")])
    assert r.returncode == 0, r.stderr[-2000:]
    recs = [json.loads(l) for l in open(log)]
    assert any(rec.get("event") == "epoch" and rec["steps"] == 6 for rec in recs)
    assert (tmp_path / "ck" / "stage0of1.pt").exists()


def test_resume_continues_the_same_run(tmp_path):
    """6 steps in one go == 4 steps, checkpoint, resume to step 6: same global step, same position in the data, same
    weights (the CPU path is bit-deterministic); a resume under a different learning rate is refused."""
    import torch

    base = ["train.py", "--device", "cpu", "--no-eval", "--synthetic"]
    r = _run(base + ["--steps", "6", "--save", str(tmp_path / "full")])
    assert r.returncode == 0, r.stderr[-2000:]
    r = _run(base + ["--steps", "4", "--save", str(tmp_path / "part")])
    assert r.returncode == 0, r.stderr[-2000:]
    r = _run(base + ["--steps", "6", "--resume", str(tmp_path / "part"), "--save", str(tmp_path / "resumed")])
    assert r.returncode == 0, r.stderr[-2000:]
    a = torch.load(tmp_path / "full" / "stage0of1.pt")
    b = torch.load(tmp_path / "resumed" / "stage0of1.pt")
    assert a["step"] == b["step"] == 6 and a["hparams"] == b["hparams"]
    assert torch.equal(a["weights"], b["weights"])
    r = _run(base + ["--steps", "6", "--resume", str(tmp_path / "part"), "--lr", "0.5"])
    assert r.returncode != 0 and "checkpoint was written with lr" in (r.stderr + r.stdout)


def test_train_accepts_reference_flags_and_pipedream():
    # same three flags as the reference CLI; 'pipedream' (a stub there) works here
    r = _run(["train.py", "--device", "cpu", "--spawn", "--dp", "2", "--pp", "2", "--schedule", "pipedream", "--steps", "3",
              "--no-eval", "--synthetic"])
    assert r.returncode == 0, r.stderr[-2000:]


def test_train_rejects_bad_grids():
    r = _run(["train.py", "--device", "cpu", "--dp", "3", "--steps", "1", "--no-eval", "--synthetic"])
    assert r.returncode != 0            # 128 % 3 != 0 / world size mismatch


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "shallowspeed", "pipe.py")),
                    reason="original project not installed in oracle/_ref (build() installs it from a checkout)")
def test_bench_reference_arm_json_contract():
    r = _run(["bench.py", "--impl", "reference", "--steps", "5", "--warmup", "3"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "dtype", "data", "config", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 5 and d["value"] > 0
    assert d["config"]["global_batch"] == 128 and d["config"]["n_mubatches"] == 4


@pytest.mark.gpu
@pytest.mark.parametrize("model,budget", [([], None), (["--hidden", "256", "--n-layers", "4"], 50_000)])
def test_bench_dump_outputs(model, budget, tmp_path, monkeypatch, capsys):
    """bench.py --dump-outputs, run in this process so the trainer can be watched: the trainer takes exactly the
    warm-up and timed steps --warmup / --steps / --repeats ask for, and the files hold its loss and parameters after
    the last of them - in full, or (over the size budget) at the documented seeded sample of each weight matrix."""
    import numpy as np

    sys.path.insert(0, ROOT)
    try:
        import bench
    finally:
        sys.path.remove(ROOT)
    from shallowspeed_b200.layers import MLP
    from shallowspeed_b200.parallel.engine import Trainer

    trainers = {}
    step_async = Trainer.step_async

    def counting_step_async(self, x, y):
        trainers[self] = trainers.get(self, 0) + 1
        return step_async(self, x, y)

    monkeypatch.setattr(Trainer, "step_async", counting_step_async)
    monkeypatch.delenv("SSB_COMM_TIMING", raising=False)
    if budget:
        monkeypatch.setattr(bench, "DUMP_BUDGET", budget)
    out = tmp_path / "dump"
    steps, warmup, repeats = 3, 5, 2
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", str(steps), "--warmup", str(warmup), "--repeats", str(repeats),
                                      "--no-alt", "--pool-batches", "8", "--dump-outputs", str(out)] + model)
    args = bench.parse()
    bench.run_ours(args)
    d = json.loads([l for l in capsys.readouterr().out.splitlines() if l.startswith("{")][-1])
    (trainer, n_steps), = trainers.items()
    # device-timed arm, then the e2e arm: warm-up, then `repeats` blocks of one aligning + `steps` timed steps each
    assert n_steps == max(3, warmup) + max(3, warmup // 4) + 2 * repeats * (steps + 1)
    assert d["steps"] == steps and len(d["timing"]["block_ms"]) == len(d["e2e"]["block_ms"]) == repeats

    sizes = bench.layer_sizes(args)
    total = sum(i * o + o for i, o in zip(sizes[:-1], sizes[1:]))
    frac = min(1.0, bench.DUMP_BUDGET / total)
    names, nbytes = [], 0
    init = MLP(sizes, 0, 1, 128).parameters()
    arena = trainer.model.arena
    for i, (n_in, n_out) in enumerate(zip(sizes[:-1], sizes[1:])):
        w_now = arena.weight_view(i).cpu().numpy()
        if frac < 1.0:
            names.append(f"W{i}_sample.npy")
            w = np.load(out / names[-1])
            idx = np.sort(np.random.RandomState(i).randint(0, n_out * n_in, int(frac * n_out * n_in)))
            assert w.shape == idx.shape and np.array_equal(w, w_now.reshape(-1)[idx])
        else:
            names.append(f"W{i}.npy")
            w = np.load(out / names[-1])
            assert w.shape == (n_out, n_in) and np.array_equal(w, w_now)
            assert not np.array_equal(w, init[2 * i].data.numpy())      # trained, not the initial weights
        names.append(f"b{i}.npy")
        b = np.load(out / names[-1])
        assert b.shape == (n_out,) and np.array_equal(b, arena.bias_view(i).reshape(-1).cpu().numpy())
        assert w.dtype == b.dtype == np.float32 and np.isfinite(w).all()
        nbytes += w.nbytes + b.nbytes
    loss = np.load(out / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == (1,) and loss[0] == np.float32(trainer.loss()) == np.float32(d["config"]["last_loss"])
    assert sorted(p.name for p in out.iterdir()) == sorted(names + ["loss.npy"])
    assert nbytes <= 4 * (bench.DUMP_BUDGET + sum(sizes[1:]))


def test_blocking_ddp_contrast_script(tmp_path):
    """scripts/ddp_blocking_mnist.py (reference: scripts/DDP_PyTorch_MNIST.py): 1 process, then 2 gloo ranks with a
    blocking all-reduce per parameter; hashes agree across ranks and the divergence from the 1-process model is reported."""
    script = os.path.join(ROOT, "scripts", "ddp_blocking_mnist.py")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    common = ["--epochs", "1", "--samples", "1280", "--device", "cpu"]
    r = subprocess.run([sys.executable, script] + common, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert (tmp_path / "data" / "models" / "model_p1.pkl").exists()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29671", script] + common, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("L1 divergence")]
    assert line and float(line[0].rsplit(" ", 1)[1]) < 1.0      # same global batches, summation order differs


def test_parsers_know_the_runtime_knobs():
    sys.path.insert(0, ROOT)
    try:
        import bench
        import train
    finally:
        sys.path.remove(ROOT)
    a = train.build_parser().parse_args(["--dp", "2", "--pp", "2", "--schedule", "pipedream-flush", "--comm", "nvls",
                                         "--pp-transport", "peer", "--watchdog-s", "30", "--precision", "tf32"])
    assert (a.comm, a.pp_transport, a.watchdog_s, a.precision, a.schedule) == ("nvls", "peer", 30.0, "tf32", "pipedream-flush")
    d = train.build_parser().parse_args([])
    assert (d.dp, d.pp, d.schedule, d.comm, d.pp_transport, d.watchdog_s, d.precision) == (1, 1, "naive", "fused", None, None, "fp32")
    old = sys.argv
    try:
        sys.argv = ["bench.py"]
        b = bench.parse()
    finally:
        sys.argv = old
    assert b.gpus == 1 and b.impl in ("ours", None, "") or b.impl == "ours"
    assert b.precision == "fp32" and b.comm == "fused" and b.pp_transport is None and not b.no_alt


def test_tuning_file_ships_with_every_variant_off_and_env_wins(tmp_path, monkeypatch):
    import json

    import shallowspeed_b200 as pkg

    cfg = json.load(open(os.path.join(ROOT, "shallowspeed_b200", "tuning.json")))
    # a switch is flipped only together with its measurement: every enabled one is named in profiles/variants_r2.md
    notes = open(os.path.join(ROOT, "profiles", "variants_r2.md")).read()
    assert all(k in notes for k, v in cfg.items() if k.startswith("SSB_") and v), "flip a switch only together with its measurement"
    assert pkg.TUNING == {} or all(k in os.environ for k in pkg.TUNING)
    # semantics of the loader, on a scratch copy
    import importlib.util

    src = open(os.path.join(ROOT, "shallowspeed_b200", "__init__.py")).read().split("TUNING = _apply_tuning()")[0]
    scratch = tmp_path / "pkgcopy"
    scratch.mkdir()
    (scratch / "__init__.py").write_text(src.replace("from . import", "# from . import"))
    (scratch / "tuning.json").write_text(json.dumps({"SSB_DEMO_ON": True, "SSB_SPLITK": 4, "SSB_DEMO_OFF": False, "other": 1}))
    monkeypatch.delenv("SSB_DEMO_ON", raising=False)
    monkeypatch.setenv("SSB_SPLITK", "2")
    monkeypatch.delenv("SSB_DEMO_OFF", raising=False)
    spec = importlib.util.spec_from_file_location("pkgcopy", scratch / "__init__.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    applied = mod._apply_tuning()
    try:
        assert applied == {"SSB_DEMO_ON": "1", "SSB_SPLITK": "2"} and "SSB_DEMO_OFF" not in os.environ
    finally:
        os.environ.pop("SSB_DEMO_ON", None)        # set by the loader itself, not by monkeypatch
