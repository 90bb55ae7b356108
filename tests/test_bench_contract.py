"""bench.py's reference arm runs without a GPU (host-generated R-MAT at a scale the host can
build), prints ONE JSON line with the contract keys, and exits 0 on non-zero ranks without work.
--dump-outputs writes the iterate of the last timed step (GPU) as a fixed sample (CPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, env=env,
                       timeout=600)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GFLOP/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("SpMV GFLOP/s") and d["steps"] == 2 and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--gpus", "2", "--steps", "2", "--warmup", "1"], capture_output=True,
                       text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_own_arm_refuses_to_run_without_a_gpu():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode != 0 and "no CPU path" in (r.stderr + r.stdout)


def test_dump_outputs_samples_a_large_x_the_same_way_every_time(tmp_path):
    torch = pytest.importorskip("torch")
    import bench
    k = bench.DUMP_X_BYTES // 8
    n = 3 * k + 5
    x = torch.arange(n, dtype=torch.float64)                # x[i] = i: the sample shows its indices
    bench.dump_outputs(str(tmp_path / "a"), x, 2.5)
    bench.dump_outputs(str(tmp_path / "b"), x, 2.5)
    a = np.load(tmp_path / "a" / "x.npy")
    assert a.dtype == np.float64 and a.shape == (k,)
    assert np.array_equal(a, np.load(tmp_path / "b" / "x.npy"))
    lo = np.arange(k, dtype=np.int64) * n // k               # one entry from every stratum
    hi = np.append(lo[1:], n)
    assert np.all(a >= lo) and np.all(a < hi)
    assert np.load(tmp_path / "a" / "eigen_estimate.npy").tolist() == [2.5]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    # a small x is written whole, in its own dtype
    bench.dump_outputs(str(tmp_path / "c"), torch.arange(1000, dtype=torch.float32) - 0.5, 1.0)
    c = np.load(tmp_path / "c" / "x.npy")
    assert c.dtype == np.float32 and np.array_equal(c, np.arange(1000, dtype=np.float32) - 0.5)


@pytest.mark.gpu
def test_dump_outputs_is_the_iterate_of_the_last_timed_step(tmp_path):
    """The own arm at R-MAT scale 14: the dumped x and ||A x|| are those of step warmup + steps of
    the same power iteration run here, for two values of --steps.  This pins what is dumped and
    when; that the iterates themselves are right is checked against the fp64 oracle by
    test_power_gpu.py and by the benchmark's own parity leg."""
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import bench
    from spmv_samples_b200 import generate
    from spmv_samples_b200.dist import PowerIteration, shard_rows

    scale, warmup = 14, 3
    dumps = {}
    for steps in (2, 3):
        out = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--override", str(scale),
                            "--steps", str(steps), "--warmup", str(warmup), "--no-configs",
                            "--no-cpu-baseline", "--e2e-steps", "0", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert line["steps"] == steps and line["warmup"] == warmup
        x = np.load(out / "x.npy")
        eig = np.load(out / "eigen_estimate.npy")
        assert x.dtype == np.float32 and x.shape == (1 << scale,) and eig.dtype == np.float64
        assert eig.tolist() == [line["config"]["eigen_estimate"]]
        dumps[warmup + steps] = (x, float(eig[0]))
    m = generate.make_config("c5", bench.SEED, scale_override=scale)
    it = PowerIteration(shard_rows(m, 0, 1), m.n_rows)
    for k in range(1, max(dumps) + 1):
        it.step()
        if k in dumps:
            x, eig = dumps[k]
            want = it.current_x().cpu().numpy()
            assert np.linalg.norm(x - want) <= 1e-6 * np.linalg.norm(want), k
            assert abs(eig - it.eigen_estimate()) <= 1e-6 * eig, k
    it.close()
    a, b = (dumps[k][0] for k in sorted(dumps))
    assert np.linalg.norm(a - b) > 1e-4 * np.linalg.norm(b)   # one more step is seen in the dump
