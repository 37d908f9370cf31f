"""bench.py interface checks: the reference arm (the oracle port timed on the host cores) prints ONE JSON line with the keys
a results reader expects, under a multi-rank launch only rank 0 works, bad arguments are refused, and --dump-outputs
writes what the last timed step computed (that one needs a GPU)."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ, OMP_NUM_THREADS="4", **(extra_env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line_on_the_host():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ToMe-transformer train samples/sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("octo_small")


def test_reference_arm_other_ranks_exit_without_work():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"],
                                  ["--microbench", "--dump-outputs", "d"]])
def test_bad_arguments_are_refused_before_any_work(args, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=tmp_path,
                       timeout=120)
    assert r.returncode == 2 and r.stdout == "" and "error" in r.stderr, r.stderr
    assert not os.listdir(tmp_path)


def test_step_outputs_are_float32_and_sample_large_arrays_at_fixed_positions():
    import torch
    import bench
    n = bench.DUMP_SAMPLE + 7
    eng = types.SimpleNamespace(loss=torch.arange(5.0), head_out=None, readout=torch.ones(2, 3, 4, dtype=torch.float64),
                                params=torch.arange(n, dtype=torch.float32), grads=-torch.arange(n, dtype=torch.float32))
    a, b = bench.step_outputs(eng), bench.step_outputs(eng)
    assert set(a) == {"loss", "readout", "params_sample", "grads_sample"}
    assert all(v.dtype == np.float32 for v in a.values())
    np.testing.assert_array_equal(a["loss"], np.arange(5.0))
    assert a["readout"].shape == (2, 3, 4)
    assert a["params_sample"].shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(a["params_sample"]) > 0)   # distinct, in order
    np.testing.assert_array_equal(a["params_sample"], b["params_sample"])
    np.testing.assert_array_equal(a["grads_sample"], -a["params_sample"])   # the same positions in every array of one size


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step_and_repeat(tmp_path):
    """Two runs with the same arguments write the same arrays (seeded inputs, seeded sample positions); loss[0] is the loss the
    JSON line reports for the timed steps; --steps sets the timed steps (the launch count of 2 steps is twice that of 1)."""
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")

    def run(steps, d):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                            "--batch", "16", "--from-pixels", "off", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, cwd=ROOT, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        return json.loads(r.stdout.strip().splitlines()[-1])

    a = run(2, tmp_path / "a")
    b = run(2, tmp_path / "b")
    one = run(1, tmp_path / "c")
    assert a["steps"] == 2 and one["steps"] == 1 and a["gpu_launches"] == 2 * one["gpu_launches"]
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) == ["grads_sample.npy", "head_out.npy", "loss.npy", "params_sample.npy",
                                                            "readout.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    arr = {n: (np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)) for n in names}
    for n, (x, y) in arr.items():
        assert x.dtype == np.float32 and x.shape == y.shape and np.isfinite(x).all(), n
        err = np.abs(x.astype(np.float64) - y).max()
        print(n, x.shape, "max |run a - run b| =", err)
        assert err <= 1e-5 * max(1.0, float(np.abs(y).max())), (n, err)
    loss = arr["loss.npy"][0]
    assert loss.shape == (17,) and loss[0] == np.float32(a["loss"])
    assert arr["head_out.npy"][0].shape == (16, 1, 8) and arr["readout.npy"][0].shape == (16, 8, 384)
