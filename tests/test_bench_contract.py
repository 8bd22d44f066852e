"""CPU: the bench.py contract that can be checked without a GPU -- the reference arm (the numpy restatement of the
reference's CPU path) prints exactly one JSON line with the keys the driver reads, and the B200 arm fails loudly
(no CPU fallback) when there is no device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = run_bench("--impl", "reference", "--config", "c1", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and d["higher_is_better"] is True
    assert d["value"] > 0 and d["unit"] == "sequences/s" and "workload" in d["config"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == pytest.approx(d["value"])
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == pytest.approx(d["value"])


def test_b200_arm_without_a_gpu_fails_loudly():
    import ctypes
    try:
        n = ctypes.CDLL("libcuda.so.1").cuInit(0)
    except OSError:
        n = 1
    if n == 0:
        pytest.skip("a CUDA device is present")
    r = run_bench("--config", "c1", "--steps", "1", "--warmup", "1")
    assert r.returncode != 0
    assert "NOGPU" in r.stderr or "no CUDA device" in r.stderr
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_samples_what_does_not_fit_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 64 * 1024)
    big = np.arange(20000, dtype=np.float32).reshape(200, 100)
    small = np.ones((2, 5), np.float32)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), 1.5, ["l0.W", "out.b"], [big, small])
    assert sorted(os.listdir(tmp_path / "a")) == ["cost.npy", "param_00_l0.W.sample.npy", "param_01_out.b.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 1024
    s = np.load(tmp_path / "a" / "param_00_l0.W.sample.npy")
    assert s.dtype == np.float32 and 0 < s.size < big.size and np.isin(s, big).all()
    np.testing.assert_array_equal(s, np.load(tmp_path / "b" / "param_00_l0.W.sample.npy"))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "param_01_out.b.npy"), small)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "cost.npy"), np.array([1.5]))


@pytest.mark.gpu
def test_b200_arm_times_the_asked_steps_and_dumps_the_state_they_leave(tmp_path):
    """The dump is the state after W warm-up steps, one untimed pass over the timed batches and the K timed steps:
    a replay of exactly those steps through train_step_cce gives the same cost and parameters."""
    import numpy as np
    import bench
    K, W = 4, 3
    out = tmp_path / "out"
    r = run_bench("--config", "c1", "--steps", str(K), "--warmup", str(W), "--no-cpu-baseline", "--dump-outputs", str(out))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "b200" and d["steps"] == K
    cost = np.load(out / "cost.npy")
    assert cost.dtype == np.float64 and cost.shape == (1,) and cost[0] == pytest.approx(d["last_cost"], abs=1e-6)

    cfg = bench.CONFIGS["c1"]
    ds = bench.make_dataset(cfg)
    pred = bench.make_predictor(cfg, ds)
    try:
        batches = bench.make_batches(pred, ds, W + K)
        for i in list(range(W + K)) + bench.timed_batches(W, K):
            X, mask, Y, pop, _ = batches[i]
            c = pred.engine.train_step_cce(X, mask, Y, pop)
        assert abs(float(c) - cost[0]) < 1e-5
        names = [n for n, _ in pred.engine.param_infos()]
        for i, (name, v) in enumerate(zip(names, pred.engine.get_all_param_values())):
            got = np.load(out / ("param_%02d_%s.npy" % (i, name)))
            assert got.dtype == np.float32 and got.shape == v.shape
            assert np.abs(got - v).max() < 1e-5, name
    finally:
        pred.engine.close()


@pytest.mark.gpu
def test_b200_arm_launches_exactly_the_kernels_of_the_asked_steps():
    """gpu_launches counts the launches of the timed region: K steps launch K times what one step does, also when K
    exceeds MAX_BATCHES and the timed steps cycle over the staged batches."""
    import bench
    K = bench.MAX_BATCHES + 5
    runs = {}
    for k in (1, K):
        r = run_bench("--config", "c1", "--steps", str(k), "--warmup", "3", "--no-cpu-baseline")
        assert r.returncode == 0, r.stderr[-2000:]
        runs[k] = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert runs[1]["gpu_launches"] > 0
    assert runs[K]["gpu_launches"] == K * runs[1]["gpu_launches"]
    assert runs[K]["steps"] == K


def test_timed_steps_cycle_over_at_most_max_batches():
    import bench
    W = 3
    assert bench.timed_batches(W, 4) == [3, 4, 5, 6]
    idx = bench.timed_batches(W, 2 * bench.MAX_BATCHES + 1)
    assert len(idx) == 2 * bench.MAX_BATCHES + 1
    assert sorted(set(idx)) == list(range(W, W + bench.MAX_BATCHES)) and idx[-1] == W
