"""The reference's own pose code as recorded in tests/golden/ref_outputs.npz.

oracle/_ref/libplstvo_ref.so (oracle/make_ref.py) is compiled from the original project's sources, which a checkout of this
repository does not contain.  tests/golden/make_ref_golden.py runs the tests that compare with it once against the real
library and stores, test by test, what every call returned.  Here `Replay` stands in for oracle.ref.Ref: each test builds
its inputs exactly as before and gets the recorded outputs back in call order, so the comparisons with the oracle and the
GPU path run on any machine.  A test whose inputs or calls change has to be re-recorded.
"""
from __future__ import annotations

import io
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")
_KINDS = {np.ndarray: 0, float: 1, int: 2, bool: 3}
_UNKIND = {1: float, 2: int, 3: bool}
_store = None


def test_key(node) -> str:
    return f"{node.module.__name__}::{node.name}"


def encode(calls) -> dict:
    """[(method name, returned value)] -> the arrays stored under one test's key."""
    blob, layout, kinds = io.BytesIO(), [], []
    for _, value in calls:
        leaves = value if isinstance(value, tuple) else (value,)
        layout.append(len(value) if isinstance(value, tuple) else -1)
        for v in leaves:
            kinds.append(_KINDS[type(v)])
            np.lib.format.write_array(blob, np.asarray(v), allow_pickle=False)
    return {"names": np.array([n for n, _ in calls]), "layout": np.array(layout, np.int32),
            "kinds": np.array(kinds, np.int8), "blob": np.frombuffer(blob.getvalue(), np.uint8)}


def decode(names, layout, kinds, blob):
    f = io.BytesIO(blob.tobytes())
    it = iter(kinds)

    def leaf():
        a = np.lib.format.read_array(f, allow_pickle=False)
        k = int(next(it))
        return a if k == 0 else _UNKIND[k](a.item())
    return [(str(n), tuple(leaf() for _ in range(n_leaves)) if n_leaves >= 0 else leaf())
            for n, n_leaves in zip(names, layout)]


class Replay:
    """Returns the recorded reference outputs of one test, call by call; a call the recording does not have is an error."""

    def __init__(self, key: str):
        global _store
        if _store is None:
            _store = dict(np.load(PATH, allow_pickle=False))
        if f"{key}/names" not in _store:
            raise KeyError(f"no recorded reference outputs for {key} in {PATH} (tests/golden/make_ref_golden.py)")
        self.key = key
        self.calls = decode(*(_store[f"{key}/{k}"] for k in ("names", "layout", "kinds", "blob")))
        self.i = 0

    def __getattr__(self, name):
        def call(*args, **kw):
            assert self.i < len(self.calls), f"{self.key}: more reference calls than were recorded"
            rec, value = self.calls[self.i]
            assert rec == name, f"{self.key}: call {self.i} is {name}, the recording has {rec}"
            self.i += 1
            return value
        return call


class Recorder:
    """Wraps the real library (oracle.ref.Ref) and keeps what every call returned."""

    def __init__(self, real):
        self.real, self.calls = real, []

    def __getattr__(self, name):
        fn = getattr(self.real, name)

        def call(*args, **kw):
            value = fn(*args, **kw)
            self.calls.append((name, value))
            return value
        return call


def for_test(node):
    """The `ref` fixture's object for one test."""
    return Replay(test_key(node))
