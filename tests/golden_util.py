"""Shared helpers for the golden fixtures (tests/golden/reference_outputs.npz, made by make_golden.py
from outputs of the unmodified reference)."""
import hashlib
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REDUCE_OUT = np.dtype([("key", "<u8"), ("val", "<u8"), ("worker", "<u8")])


def golden():
    return np.load(os.path.join(HERE, "golden", "reference_outputs.npz"))


def golden_r2():
    """larger cases (digests only), made by tests/golden/make_golden_r2.py from the unmodified reference"""
    return np.load(os.path.join(HERE, "golden", "reference_outputs_r2.npz"))


def golden_live():
    """outputs of reference runs on file inputs and fresh shapes, made by tests/golden/make_golden_live.py"""
    return np.load(os.path.join(HERE, "golden", "reference_outputs_live.npz"))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# inputs of the cases in reference_outputs_live.npz (shared by the tests and make_golden_live.py)
LIVE_SORT_CASES = [(1, 30000), (2, 1), (3, 12345), (8, 200000)]       # (workers, n)
LIVE_REDUCE_ZERO_KEY_WORKERS = [1, 2, 5]
LIVE_REDUCE_TO_INDEX_CASES = [(1, 5000, 300), (2, 40000, 7001), (5, 3000, 100000)]       # (workers, n, universe)


def live_sort_input(workers, n):
    rng = np.random.RandomState(workers * 1000 + n % 997)
    return rng.randint(0, 50, size=n).astype(np.uint64) if workers == 3 else \
        rng.randint(0, 2**63, size=n).astype(np.uint64)


def live_reduce_zero_key_input(workers):
    rng = np.random.RandomState(workers)
    n = 60000
    kv = np.zeros(n, dtype=[("key", "<u8"), ("val", "<u8")])
    kv["key"] = rng.randint(0, 500, size=n)          # includes key 0: sentinel slot path
    kv["val"] = rng.randint(0, 1000, size=n)
    return kv
