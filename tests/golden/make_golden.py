#!/usr/bin/env python
"""Regenerate tests/golden/*.npz from the UNMODIFIED reference engine.

Run where the reference sources exist (oracle/Makefile, REF=<reference checkout>):
    make -C oracle ref && OMP_NUM_THREADS=1 python tests/golden/make_golden.py
The reference is only deterministic single-threaded (SURVEY.md §0 fact 2), hence OMP_NUM_THREADS=1.
Every scenario is recorded twice and must hash identically before it is written.  Last, the non-GPU suite runs with
MAGENT_B200_RECORD_REFERENCE=1, which rewrites tests/golden/reference_results.npz: the results of the reference that
the differential tests compare with (golden_common.check_reference_result).
"""
import os
import sys

os.environ["OMP_NUM_THREADS"] = "1"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import numpy as np  # noqa: E402
import parity_common as pc  # noqa: E402
import golden_common as gc  # noqa: E402

if __name__ == "__main__":
    assert os.path.exists(pc.REF_LIB), "build the reference first: make -C oracle ref"
    for name in gc.SCENARIOS:
        a, b = gc.pack(gc.record(name, pc.REF_LIB)), gc.pack(gc.record(name, pc.REF_LIB))
        assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a), name + ": reference not deterministic"
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **a)
        print("%-16s %3d steps  final num %s  %6.1f KB" % (name, int(a["n_steps"]),
              a["s%d_num" % (int(a["n_steps"]) - 1)].tolist(), os.path.getsize(path) / 1024))
    import tempfile
    a, b = gc.record_edge_cases(pc.REF_LIB, tempfile.mkdtemp()), gc.record_edge_cases(pc.REF_LIB, tempfile.mkdtemp())
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a), "edge cases: reference not deterministic"
    np.savez_compressed(gc.EDGE_FILE, **a)
    print("edge_cases       %s" % sorted(a))
    import subprocess
    if os.path.exists(gc.RESULTS_FILE):
        os.remove(gc.RESULTS_FILE)
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "not gpu", os.path.dirname(HERE)],
                   env=dict(os.environ, **{gc.RECORD_ENV: "1"}), check=True)
    print("reference_results %6.1f KB" % (os.path.getsize(gc.RESULTS_FILE) / 1024))
