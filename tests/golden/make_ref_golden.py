"""Records tests/golden/ref_outputs.npz: what the reference's own pose code (oracle/_ref/libplstvo_ref.so) returned to every
test that compares with it (the `ref` fixture, tests/ref_golden.py).

Needs the library, which oracle/make_ref.py compiles from the original project's sources (PLSTVO_REFERENCE points at a
checkout of rubengooj/stvo-pl).  The tests run under pytest with the real library behind `ref`; the GPU tests among them run
with the oracle in the place of the CUDA engine (their reference calls only see inputs built on the CPU).  A failing test
writes nothing.

Usage: python tests/golden/make_ref_golden.py
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import ref_golden  # noqa: E402

TESTS = ["tests/test_oracle_ref.py",
         "tests/test_gpu_pose.py::test_explicit_lists_c5_size",
         "tests/test_gpu_parity_holes.py::test_degenerate_previous_segments_through_the_solver",
         "tests/test_gpu_parity_holes.py::test_zero_length_previous_segments",
         "tests/test_gpu_parity_holes.py::test_outlier_threshold_adversarial"]


class OracleAsEngine:
    """The engine methods those GPU tests call, answered by the oracle."""

    def __init__(self, device=-1):
        from oracle.oracle import Oracle
        self.orc = Oracle()

    def optimize_pose(self, cam, cfg, matched, priors=None):
        return self.orc.optimize_pose(cam, cfg, matched, priors)[1:]


def main():
    from oracle import make_ref
    from oracle.ref import Ref
    import stvo_pl_b200.engine
    make_ref.build()
    real, recorded = Ref(), {}

    def record(node):
        recorded[ref_golden.test_key(node)] = rec = ref_golden.Recorder(real)
        return rec
    ref_golden.for_test = record
    stvo_pl_b200.engine.Engine = OracleAsEngine
    rc = pytest.main(["-q", "-p", "no:cacheprovider", "--rootdir", ROOT] + [os.path.join(ROOT, t) for t in TESTS])
    if rc != 0:
        sys.exit(f"pytest failed ({rc}): nothing written")
    out = {}
    for key, rec in sorted(recorded.items()):
        for name, arr in ref_golden.encode(rec.calls).items():
            out[f"{key}/{name}"] = arr
    np.savez_compressed(ref_golden.PATH, **out)
    print(f"{ref_golden.PATH}: {len(recorded)} tests, {sum(len(r.calls) for r in recorded.values())} calls, "
          f"{os.path.getsize(ref_golden.PATH)} bytes")


if __name__ == "__main__":
    main()
