"""The reference's own shaders, pinned by digest — TEST INFRASTRUCTURE.

The pinning tests compare the oracle with the reference's shaders (tests/refglsl.py) bit for bit.  Those shaders are built from the
reference's GLSL, which is not part of this repository, so what they computed is stored instead: tests/golden/make_golden.py runs each
pinning case once on the shaders through `Record`, which logs, for every pass call in order, a digest of the call's inputs and a digest of
each output (tests/golden/reference_pins.json).  The tests run the same case through `Replay`, which executes every call on the oracle
(tests/orc.py) and requires the same digests: a differing byte in any output of any pass fails at the call that produced it.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os

import numpy as np

PINS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.json")


def digest(*objs) -> str:
    """SHA-256 (first 16 hex digits) over the bytes of arrays, ctypes structures and scalars, in order.  Other objects (orc.Env) are
    skipped: they are built from arrays that are hashed where they enter."""
    h = hashlib.sha256()

    def feed(x):
        if isinstance(x, (tuple, list)):
            for y in x:
                feed(y)
            return
        if isinstance(x, np.ndarray):
            b = np.ascontiguousarray(x).tobytes()
        elif isinstance(x, C.Structure):
            b = bytes(x)
        elif isinstance(x, np.generic):
            b = x.tobytes()
        elif x is None or isinstance(x, (bool, int, float, str)):
            b = repr(x).encode()
        else:
            return
        h.update(len(b).to_bytes(8, "little"))
        h.update(b)

    feed(objs)
    return h.hexdigest()[:16]


def _outputs(r) -> list:
    return [digest(x) for x in (r if isinstance(r, tuple) else (r,))]


def load(case: str):
    with open(PINS) as f:
        return json.load(f)[case]


class Record:
    """Runs the passes on `impl` (tests/refglsl.py) and logs [pass, inputs digest, output digests] per call."""

    def __init__(self, impl):
        self.impl, self.log = impl, []

    def __getattr__(self, name):
        fn = getattr(self.impl, name)

        def call(*a, **kw):
            r = fn(*a, **kw)
            self.log.append([name, digest(a, sorted(kw.items())), _outputs(r)])
            return r

        return call


class Replay:
    """Runs the passes on the oracle and checks every call against the reference's log of `case`."""

    def __init__(self, case: str):
        import orc

        self.case, self.impl, self.log, self.n = case, orc, load(case), 0

    def __getattr__(self, name):
        fn = getattr(self.impl, name)

        def call(*a, **kw):
            i = self.n
            assert i < len(self.log), f"{self.case}: more pass calls than the reference's run made ({len(self.log)})"
            want_name, want_in, want_out = self.log[i]
            where = f"{self.case}, call {i} ({name})"
            assert name == want_name, f"{where}: the reference's run called {want_name} here"
            assert digest(a, sorted(kw.items())) == want_in, f"{where}: not the inputs the reference's shaders were run on"
            r = fn(*a, **kw)
            got = _outputs(r)
            bad = [j for j, (g, w) in enumerate(zip(got, want_out)) if g != w]
            assert len(got) == len(want_out) and not bad, f"{where}: output(s) {bad} differ from the reference's shaders"
            self.n += 1
            return r

        return call

    def finish(self):
        assert self.n == len(self.log), f"{self.case}: {self.n} pass calls, the reference's run made {len(self.log)}"
