#!/usr/bin/env python
"""Fixtures tests/golden/reference_outputs_live.npz: outputs of the UNMODIFIED reference (oracle/_ref/thrill_ref_driver) on
file inputs and on fresh shapes, which test_oracle_golden.py's test_live_reference_* compare the oracle against.  Sort
outputs are stored as digests, reduce outputs in full.  Needs oracle/_ref (make -C oracle ref):
python tests/golden/make_golden_live.py"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as O  # noqa: E402
from golden_util import (LIVE_REDUCE_TO_INDEX_CASES, LIVE_REDUCE_ZERO_KEY_WORKERS, LIVE_SORT_CASES, REDUCE_OUT,  # noqa: E402
                         live_reduce_zero_key_input, live_sort_input, sha)


def main():
    assert O.have_ref_driver(), "build oracle/_ref first: make -C oracle ref"
    g = {}
    with tempfile.TemporaryDirectory() as d:
        inp, out = os.path.join(d, "in.bin"), os.path.join(d, "o.bin")
        for workers, n in LIVE_SORT_CASES:
            live_sort_input(workers, n).tofile(inp)
            O.run_ref_driver(workers=workers, op="sort_u64", gen="file", out=out, **{"in": inp})
            a = np.fromfile(out, dtype=np.uint64)
            assert len(a) == n
            g["sort_file_w%d_n%d_sha256" % (workers, n)] = np.array(sha(a))
        for workers in LIVE_REDUCE_ZERO_KEY_WORKERS:
            live_reduce_zero_key_input(workers).tofile(inp)
            O.run_ref_driver(workers=workers, op="reduce_u64", gen="file", out=out, **{"in": inp})
            g["reduce_u64_zero_key_w%d" % workers] = np.sort(np.fromfile(out, dtype=REDUCE_OUT), order="key")
        for workers, n, universe in LIVE_REDUCE_TO_INDEX_CASES:
            O.run_ref_driver(workers=workers, op="reduce_to_index", gen="uniform", universe=universe, n=n, exact=1, out=out)
            g["reduce_to_index_uniform_u%d_%d_exact1_w%d" % (universe, n, workers)] = np.fromfile(out, dtype=O.KV)
    np.savez_compressed(os.path.join(HERE, "reference_outputs_live.npz"), **g)
    print("wrote reference_outputs_live.npz", {k: (str(v) if v.ndim == 0 else v.shape) for k, v in g.items()})


if __name__ == "__main__":
    main()
