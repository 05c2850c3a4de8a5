"""CPU: the JSON contract of bench.py's reference arm (the CPU restatement of the learner step timed on the host cores) and
the workload description shared by both arms -- without running a full 512-transition step (the timed function is stubbed)."""
import json
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def test_reference_arm_line(capsys, monkeypatch):
    import bench
    calls = []

    def fake_learner(batch, threads=None):
        calls.append(batch)
        return lambda i: None

    monkeypatch.setattr(bench, "oracle_learner", fake_learner)
    monkeypatch.setattr(bench, "best_threads", lambda: 4)
    monkeypatch.setenv("RANK", "0")
    args = types.SimpleNamespace(gpus=2, steps=3, warmup=1, replay_capacity=1 << 19)
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["n_gpus"] == 2 and line["steps"] == 3
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["value"] == line["value"]
    # both arms describe the workload with the same keys / values (the driver compares them)
    assert line["config"] == bench.config_dict(2, 1 << 19)
    assert set(bench.config_dict(1, 1 << 19)) == set(line["config"])
    # other ranks of a torchrun launch leave without work and without output
    monkeypatch.setenv("RANK", "1")
    bench.run_reference(args)
    assert capsys.readouterr().out == ""


def test_dump_outputs_files(tmp_path):
    import numpy as np
    import pytest
    import bench
    d = str(tmp_path / "out")
    idx, loss = np.arange(512, dtype=np.float64) + 2 ** 40, np.linspace(0, 1, 512, dtype=np.float32)
    bench.dump_outputs(d, {"tree_idxs": idx, "loss": loss})
    assert sorted(os.listdir(d)) == ["loss.npy", "tree_idxs.npy"]
    assert np.array_equal(np.load(os.path.join(d, "tree_idxs.npy")), idx)
    got = np.load(os.path.join(d, "loss.npy"))
    assert got.dtype == np.float32 and np.array_equal(got, loss)
    with pytest.raises(AssertionError):
        bench.dump_outputs(d, {"tree_idxs": idx.astype(np.int64)})


def test_bench_argument_checks(monkeypatch, tmp_path):
    import pytest
    import bench
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                 ["--gpus", "2", "--topology", "apex", "--dump-outputs", str(tmp_path)]):
        monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
        with pytest.raises(SystemExit) as e:
            bench.main()
        assert e.value.code == 2, argv
    assert not os.listdir(tmp_path)
