"""bench.py's command-line contract, as far as it can be checked without a GPU: the reference arm (the unmodified reference on
the host cores) prints one JSON line with the keys the driver reads, on the same `config` object our arm would print; our arm
refuses to run without a GPU (no CPU fallback); --dump-outputs writes exact, reproducible files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.ref
@pytest.mark.parametrize("metric,nflag,unit", [("sort", "--n", "keys/s"), ("reduce", "--reduce-n", "records/s")])
def test_reference_arm_prints_the_contract_line(metric, nflag, unit):
    if not O.have_ref_driver():
        pytest.skip("oracle/_ref/thrill_ref_driver not built")
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--metric", metric, "--gpus", "2",
           "--steps", "1", "--warmup", "1", nflag, "200000"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, RANK="0"))
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "config", "cpu_baseline", "e2e", "dtype", "data"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == unit and line["n_gpus"] == 2 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    # the same config object as our arm prints for this metric / size / worker count (the driver compares them)
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.workload_config(metric, 200000, 2)
    # the other ranks of a torchrun launch exit without work
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=60, env=dict(os.environ, RANK="1"))
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_our_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--n", "1000"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode != 0 and "no CPU fallback" in (res.stderr + res.stdout)


def test_write_outputs_files_dtypes_sampling_and_exact_key_halves(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(7)
    n = bench.DUMP_ITEMS + 12345
    keys = np.sort(rng.integers(0, 2**64 - 1, size=n, dtype=np.uint64, endpoint=True))
    bench.write_outputs(str(tmp_path / "a"), "sort", 1, 0, keys)
    bench.write_outputs(str(tmp_path / "b"), "sort", 1, 0, keys.copy())
    names = sorted(os.listdir(str(tmp_path / "a")))
    assert names == ["sort_count.npy", "sort_index.npy", "sort_keys_hi32.npy", "sort_keys_lo32.npy"]
    got = {}
    for f in names:
        a, b = np.load(str(tmp_path / "a" / f)), np.load(str(tmp_path / "b" / f))
        assert a.dtype == np.float64 and np.array_equal(a, b), f          # same output, same files
        got[f[len("sort_"):-len(".npy")]] = a
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in names) <= 64 << 20
    assert got["count"].tolist() == [n]
    idx = got["index"].astype(np.int64)
    assert len(idx) == bench.DUMP_ITEMS and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n
    hi, lo = got["keys_hi32"].astype(np.uint64), got["keys_lo32"].astype(np.uint64)
    assert np.array_equal((hi << np.uint64(32)) | lo, keys[idx])       # the float64 halves are exact
    # an output smaller than the per-rank share is written whole; ranks of a multi-GPU job get their own files
    k = np.arange(1000, dtype=np.uint64) << np.uint64(40)
    v = rng.random(1000)
    bench.write_outputs(str(tmp_path / "c"), "reduce", 2, 1, k, v)
    assert sorted(os.listdir(str(tmp_path / "c"))) == ["reduce_%s_rank1.npy" % f for f in
                                                       ("count", "index", "keys_hi32", "keys_lo32", "vals")]
    assert np.array_equal(np.load(str(tmp_path / "c" / "reduce_index_rank1.npy")), np.arange(1000))
    assert np.array_equal(np.load(str(tmp_path / "c" / "reduce_vals_rank1.npy")), v)
    assert np.array_equal(np.load(str(tmp_path / "c" / "reduce_keys_hi32_rank1.npy")).astype(np.uint64) << np.uint64(32), k)


@pytest.mark.parametrize("flags,msg", [(["--impl", "reference", "--dump-outputs", "d"], "--dump-outputs"),
                                       (["--steps", "0"], "--steps")])
def test_flags_the_bench_cannot_honour_are_refused(tmp_path, flags, msg):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + flags, capture_output=True, text=True,
                         timeout=120, cwd=str(tmp_path))
    assert res.returncode == 2 and msg in res.stderr and not os.listdir(str(tmp_path))
