"""Pins oracle/thrill_oracle.c against outputs of the UNMODIFIED reference:
(1) the committed fixtures tests/golden/reference_outputs.npz (made by tests/golden/make_golden.py),
(2) tests/golden/reference_outputs_live.npz (made by tests/golden/make_golden_live.py), the reference's runs on file
inputs and fresh shapes.
CPU only."""
import os

import numpy as np
import pytest

import oracle_lib as O
from golden_util import (LIVE_REDUCE_TO_INDEX_CASES, LIVE_REDUCE_ZERO_KEY_WORKERS, LIVE_SORT_CASES, golden, golden_live,
                         golden_r2, live_reduce_zero_key_input, live_sort_input, sha)


def _counts(n, p):
    c = np.full(p, n // p, dtype=np.uint64)
    c[: n % p] += 1
    return c


def test_golden_sort_uniform():
    g = golden()
    keys = O.gen_sort_uniform(0, 4096)
    out, _ = O.sort_operator(keys, _counts(4096, 3))
    assert np.array_equal(out.view(np.uint64), g["sort_uniform_4096_w3"])
    keys = O.gen_sort_uniform(0, 1000000)
    out, _ = O.sort_operator(keys, _counts(1000000, 4))
    assert sha(out) == str(g["sort_uniform_1000000_w4_sha256"])


def test_golden_sort_zipf_duplicates():
    g = golden()
    cdf = O.zipf_cdf(1024)
    keys = O.gen_sort_zipf(0, 50000, cdf)
    out, oc = O.sort_operator(keys, _counts(50000, 5))
    out = out.view(np.uint64)
    assert np.array_equal(out[:64], g["sort_zipf_u1024_50000_w5_head"])
    assert sha(out) == str(g["sort_zipf_u1024_50000_w5_sha256"])


def test_golden_reduce_f64_zipf_tolerance_and_ownership():
    g = golden()
    ref = g["reduce_f64_zipf_u4096_200000_w3"]
    cdf = O.zipf_cdf(4096)
    kv = O.gen_reduce_zipf(0, 200000, cdf)
    out, oc = O.reduce_operator(kv, _counts(200000, 3), 64 << 20, O.OP_SUM_F64)
    owner = np.repeat(np.arange(3, dtype=np.uint64), oc.astype(np.int64))
    order = np.argsort(out["key"], kind="stable")
    out, owner = out[order], owner[order]
    assert np.array_equal(out["key"], ref["key"])
    # same owner worker as the reference: key -> Hash128to64(0,key) % p
    assert np.array_equal(owner, ref["worker"])
    a, b = out["val"].view(np.float64), ref["val"].view(np.float64)
    assert np.all(np.abs(a - b) <= 1e-9 * np.maximum(1.0, np.abs(b)))      # SURVEY.md §8d tolerance


def test_golden_reduce_exact_modes_bit_identical():
    g = golden()
    ref = g["reduce_f64_exact_zipf_u4096_200000_w4"]
    cdf = O.zipf_cdf(4096)
    kv = O.gen_reduce_zipf(0, 200000, cdf, exact=1)
    out, oc = O.reduce_operator(kv, _counts(200000, 4), 64 << 20, O.OP_SUM_F64)
    out = np.sort(out, order="key")
    assert np.array_equal(out["key"], ref["key"]) and np.array_equal(out["val"], ref["val"])
    ref = g["reduce_u64_uniform_u3000_100000_w2"]
    kv = O.gen_reduce_uniform(0, 100000, universe=3000, exact=2)
    out, oc = O.reduce_operator(kv, _counts(100000, 2), 64 << 20, O.OP_SUM_U64)
    out = np.sort(out, order="key")
    assert np.array_equal(out["key"], ref["key"]) and np.array_equal(out["val"], ref["val"])
    # and the simple checker agrees with the faithful table restatement
    simple = O.reduce_simple(kv, O.OP_SUM_U64)
    assert np.array_equal(simple, out)


def test_golden_terasort_records():
    g = golden()
    rec = O.gen_records(0, 20000)
    out, _ = O.sort_operator(rec, _counts(20000, 3), desc=O.RECORD_DESC)
    out = out.reshape(-1, 100)
    assert np.array_equal(out[:8], g["terasort_20000_w3_head"])
    assert sha(out) == str(g["terasort_20000_w3_sha256"])


# ---- the reference's runs on file inputs and fresh shapes (outputs stored by tests/golden/make_golden_live.py) ----
@pytest.mark.parametrize("workers,n", LIVE_SORT_CASES)
def test_live_reference_sort_file_input(workers, n):
    keys = live_sort_input(workers, n)
    out, _ = O.sort_operator(keys, _counts(n, workers))
    assert sha(out.view(np.uint64)) == str(golden_live()["sort_file_w%d_n%d_sha256" % (workers, n)])


@pytest.mark.parametrize("workers", LIVE_REDUCE_ZERO_KEY_WORKERS)
def test_live_reference_reduce_with_zero_key(workers):
    kv = live_reduce_zero_key_input(workers)
    n = len(kv)
    ref = golden_live()["reduce_u64_zero_key_w%d" % workers]
    out, oc = O.reduce_operator(kv, _counts(n, workers), 64 << 20, O.OP_SUM_U64)
    owner = np.repeat(np.arange(workers, dtype=np.uint64), oc.astype(np.int64))
    order = np.argsort(out["key"], kind="stable")
    assert np.array_equal(out["key"][order], ref["key"])
    assert np.array_equal(out["val"][order], ref["val"])
    assert np.array_equal(owner[order], ref["worker"])


def _rti_input(gen, n, universe, exact):
    if gen == "zipf":
        kv = O.gen_reduce_zipf(0, n, O.zipf_cdf(universe), exact=exact)
    else:
        kv = O.gen_reduce_uniform(0, n, universe=universe, exact=exact)
    kv["key"] %= universe                      # what ref_driver's reduce_to_index op feeds ReduceToIndex
    return kv


def test_golden_reduce_to_index_dense_result():
    """ReduceToIndex (api/reduce_to_index.hpp:60-237, the PageRank step): the concatenation over the reference's workers is
    the dense array; exact-mode doubles are bit-identical, real doubles within the stated tolerance, missing indices keep
    the neutral element (0, 0.0)."""
    g = golden()
    ref = g["reduce_to_index_zipf_u1000_20000_exact1_w3"]
    out = O.reduce_to_index(_rti_input("zipf", 20000, 1000, 1), 1000, O.OP_SUM_F64)
    assert np.array_equal(out, ref)
    ref = g["reduce_to_index_zipf_u1000_20000_exact0_w4"]
    out = O.reduce_to_index(_rti_input("zipf", 20000, 1000, 0), 1000, O.OP_SUM_F64)
    assert np.array_equal(out["key"], ref["key"])
    a, b = out["val"].view(np.float64), ref["val"].view(np.float64)
    assert np.all(np.abs(a - b) <= 1e-9 * np.maximum(1.0, np.abs(b)))
    ref = g["reduce_to_index_uniform_u50000_3000_exact1_w5"]
    out = O.reduce_to_index(_rti_input("uniform", 3000, 50000, 1), 50000, O.OP_SUM_F64)
    assert np.array_equal(out, ref)
    assert np.count_nonzero((ref["key"] == 0) & (ref["val"] == 0)) > 40000        # mostly neutral


@pytest.mark.parametrize("workers,n,universe", LIVE_REDUCE_TO_INDEX_CASES)
def test_live_reference_reduce_to_index(workers, n, universe):
    """the unmodified reference's ReduceToIndex on a fresh shape (dense, sparse, more workers than data per index): the
    oracle's dense array is bit-identical in exact mode"""
    ref = golden_live()["reduce_to_index_uniform_u%d_%d_exact1_w%d" % (universe, n, workers)]
    assert len(ref) == universe
    mine = O.reduce_to_index(_rti_input("uniform", n, universe, 1), universe, O.OP_SUM_F64)
    assert np.array_equal(mine, ref)


def test_golden_r2_larger_cases_pin_the_oracle():
    """tests/golden/reference_outputs_r2.npz: TeraSort 1e6 records, Sort 1e7 uniform / 5e6 Zipf keys, ReducePair 4e6 Zipf
    records (exact mode) of the unmodified reference vs the C restatement"""
    g = golden_r2()
    rec = O.gen_records(0, 1000000)
    out = O.sort_items(rec, O.RECORD_DESC).reshape(-1, 100)
    assert np.array_equal(out[:4], g["terasort_1000000_head"]) and np.array_equal(out[-4:], g["terasort_1000000_tail"])
    assert sha(out) == str(g["terasort_1000000_sha256"])
    keys = O.gen_sort_uniform(0, 10000000)
    assert sha(O.sort_items(keys)) == str(g["sort_uniform_10000000_sha256"])
    keys = O.gen_sort_zipf(0, 5000000, O.zipf_cdf(1 << 20))
    out, _ = O.sort_operator(keys, _counts(5000000, 5))
    assert sha(out) == str(g["sort_zipf_u2^20_5000000_sha256"])
    kv = O.gen_reduce_zipf(0, 4000000, O.zipf_cdf(1 << 20), exact=1)
    red = O.reduce_simple(kv, O.OP_SUM_F64)
    assert len(red) == int(g["reduce_f64_exact_zipf_u2^20_4000000_distinct"])
    assert sha(red) == str(g["reduce_f64_exact_zipf_u2^20_4000000_sha256"])


@pytest.mark.ref
def test_cfg1_word_count_plumbing_two_loopback_workers(tmp_path):
    """BASELINE.json configs[0]: the reference's own examples/word_count on ~1 MB of synthetic text with 2 local-loopback
    workers (CPU reference, plumbing only: nothing of the GPU path is involved).  Run through oracle/_ref/thrill_ref_driver."""
    import collections
    import subprocess
    if not O.have_ref_driver():
        pytest.skip("oracle/_ref/thrill_ref_driver not built")
    env = dict(os.environ, THRILL_NET="local", THRILL_LOCAL="2", THRILL_WORKERS_PER_HOST="1", THRILL_LOG="")
    out = os.path.join(str(tmp_path), "wc.txt")
    res = subprocess.run([O.REF_DRIVER, "op=word_count", "n=15000", "out=" + out], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    line = [l for l in res.stdout.splitlines() if l.startswith("WORDCOUNT")][0]
    assert "words=150000" in line and "workers=2" in res.stdout
    counts = dict((w, int(c)) for w, c in (l.split() for l in open(out)))
    assert sum(counts.values()) == 150000 and 900 <= len(counts) <= 1000
    # the reference's own fixture (its tests/inputs/wordcount.in, checked by tests/examples/word_count_test.cpp: 71 pairs)
    sample = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wordcount.in")
    res = subprocess.run([O.REF_DRIVER, "op=word_count", "gen=file", "in=" + sample, "out=" + out], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0
    got = dict((w, int(c)) for w, c in (l.split() for l in open(out)))
    want = collections.Counter(open(sample).read().split())
    assert got == dict(want) and len(got) == 71
