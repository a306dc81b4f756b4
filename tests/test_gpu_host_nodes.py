"""The drop-in inside the unmodified reference: runs the prebuilt oracle/_ref/host/gpu_nodes_test (a real Thrill
job linking the reference library and libthrill_gpu.so) and requires every comparison of the stock CPU operator
against the GPU node to PASS.  pytest -m gpu."""
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "host", "gpu_nodes_test")


@pytest.mark.skipif(not os.path.exists(BIN), reason="oracle/_ref/host/gpu_nodes_test not built (make -C tests/host)")
def test_gpu_nodes_inside_thrill_single_worker():
    env = dict(os.environ, THRILL_NET="mock", THRILL_LOCAL="1", THRILL_WORKERS_PER_HOST="1", THRILL_LOG="")
    res = subprocess.run([BIN, "2000000"], env=env, capture_output=True, text=True, timeout=900)
    lines = [l for l in res.stdout.splitlines() if l.startswith(("PASS", "FAIL"))]
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert len(lines) == 10 and all(l.startswith("PASS") for l in lines), lines


@pytest.mark.skipif(not os.path.exists(BIN), reason="oracle/_ref/host/gpu_nodes_test not built")
def test_gpu_nodes_inside_thrill_two_workers_two_gpus():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (gpurun --gpus 2)")
    env = dict(os.environ, THRILL_NET="mock", THRILL_LOCAL="1", THRILL_WORKERS_PER_HOST="2", THRILL_LOG="")
    res = subprocess.run([BIN, "3000000"], env=env, capture_output=True, text=True, timeout=900)
    lines = [l for l in res.stdout.splitlines() if l.startswith(("PASS", "FAIL"))]
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert len(lines) == 10 and all(l.startswith("PASS") for l in lines), lines
