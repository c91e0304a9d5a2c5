"""The original C extension (WojciechMula/pyahocorasick, compiled into oracle/_ref), recorded once and replayed.

The differential tests drive the drop-in and the original side by side and compare every answer.  The original is
not part of this repository, so each such test runs against a stand-in: a module whose every call (module
attributes, Automaton methods, iterator steps, exceptions included) returns what the original returned when the same
test ran against it.  The calls are checked as they happen: each one must name the same operation with the same
arguments as when it was recorded (one byte of a digest of them, which a test that has gone its own way misses for a
call or two at most), so a test that diverges from its recording fails instead of comparing against someone else's
answer.

    python tests/golden/record_reference.py        # re-record, where oracle/_ref is built

Traces live in tests/golden/reference/<test module>.pkl.xz: {test name with parameters: [event, ...]}.
"""
from __future__ import annotations

import builtins
import hashlib
import io
import lzma
import os
import pickle

import numpy as np
import pytest

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
_REF_TYPES = {"Automaton", "AutomatonSearchIter", "AutomatonSearchIterLong", "AutomatonItemsIter"}
RECORDING = None        # set by tests/golden/record_reference.py: {module: {test: events}}


class _PlainUnpickler(pickle.Unpickler):
    """traces hold plain data only: no class may be imported while reading one"""
    def find_class(self, module, name):
        raise pickle.UnpicklingError(f"{module}.{name} in a reference trace")


def load_traces(module: str) -> dict:
    path = os.path.join(_DIR, module + ".pkl.xz")
    if not os.path.exists(path):
        return {}
    with lzma.open(path, "rb") as f:
        return _PlainUnpickler(io.BytesIO(f.read())).load()


def save_traces(module: str, traces: dict) -> None:
    os.makedirs(_DIR, exist_ok=True)
    with lzma.open(os.path.join(_DIR, module + ".pkl.xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        pickle.dump(traces, f, protocol=4)


class _Session:
    """one test's conversation with the original: a list of events (op, args digest, outcome, callbacks, file)"""

    def __init__(self, events=None):
        self.recording = events is None
        self.events = [] if events is None else events
        self.pos = 0
        self.n_objects = 0

    def norm(self, x):
        if isinstance(x, _Proxy):
            return ("ref", x._id)
        if isinstance(x, (list, tuple)):
            return type(x)(self.norm(y) for y in x)
        if isinstance(x, dict):
            return {k: self.norm(v) for k, v in x.items()}
        if isinstance(x, np.integer):
            return int(x)
        if callable(x):
            return "callable"
        return x

    def digest(self, op, args, kw):
        if op in ("save", "load"):                  # the path is the test's temporary file: what counts is its content
            path, args = args[0], args[1:]
            args = (open(path, "rb").read() if op == "load" else None,) + tuple(args)
        blob = pickle.dumps((op, self.norm(tuple(args)), self.norm(kw)), protocol=4)
        return hashlib.blake2b(blob, digest_size=1).digest()

    def outcome(self, value):
        if isinstance(value, type):
            return ("c", value.__name__)
        if type(value).__name__ in _REF_TYPES:
            return ("r", type(value).__name__)
        if isinstance(value, tuple) and value and isinstance(value[0], type):      # __reduce__: (class, args)
            return ("v", (None,) + value[1:])
        return ("v", value)

    def call(self, target, op, fn, args, kw):
        d = self.digest(op, args, kw)
        if self.recording:
            calls = []
            wrapped = [(lambda *a, _f=a: (calls.append(a), _f(*a))[1]) if callable(a) and not isinstance(a, _Proxy) else _unwrap(a)
                       for a in args]
            try:
                value = fn(*wrapped, **{k: _unwrap(v) for k, v in kw.items()})
                out = self.outcome(value)
            except Exception as e:                   # noqa: BLE001 -- the exception is the original's answer
                value, out = None, ("e", (type(e).__name__, str(e)))
            saved = open(args[0], "rb").read() if op == "save" and out[0] != "e" else None
            self.events.append((op, d, out, calls, saved))
            return self.result(out, value)
        if self.pos >= len(self.events):
            pytest.fail(f"the test calls {target}.{op}() after the end of its recording ({len(self.events)} calls)")
        rop, rd, out, calls, saved = self.events[self.pos]
        if (rop, rd) != (op, d):
            pytest.fail(f"call {self.pos} differs from the recording: {target}.{op}() with arguments {d.hex()}, "
                        f"recorded {rop}() with {rd.hex()}")
        self.pos += 1
        for a in args:                              # callbacks see what the original passed them
            if callable(a) and not isinstance(a, _Proxy):
                for c in calls:
                    a(*c)
        if saved is not None:
            with open(args[0], "wb") as f:
                f.write(saved)
        return self.result(out, None)

    def result(self, out, value):
        kind, v = out
        if kind == "e":
            raise getattr(builtins, v[0])(v[1])
        if kind == "r":
            self.n_objects += 1
            return (_Automaton if v == "Automaton" else _Iterator)(self, value, self.n_objects)
        if kind == "c":
            return f"<class {v}>"
        return v


def _unwrap(x):
    return x._obj if isinstance(x, _Proxy) else x


class _Proxy:
    """an object of the original (the module, an automaton, an iterator), live while recording, replayed otherwise"""

    def __init__(self, session, obj, ident):
        self.__dict__.update(_s=session, _obj=obj, _id=ident)

    def _call(self, op, *args, **kw):
        fn = getattr(self._obj, op) if self._s.recording else None
        return self._s.call(self._id, op, fn, args, kw)

    def __getattr__(self, name):
        s = self._s
        if s.recording:
            attr = getattr(self._obj, name)
            if not callable(attr):
                s.events.append(("." + name, b"", s.outcome(attr), [], None))
                return attr
        elif s.pos < len(s.events) and s.events[s.pos][0] == "." + name:
            s.pos += 1
            return s.result(s.events[s.pos - 1][2], None)
        return lambda *a, **kw: self._call(name, *a, **kw)


class _Iterator(_Proxy):
    def __iter__(self):
        return self

    def __next__(self):
        return self._call("__next__")


class _Automaton(_Proxy):
    def __len__(self):
        return self._call("__len__")

    def __contains__(self, x):
        return self._call("__contains__", x)

    def __reduce__(self):
        return self._call("__reduce__")


def _records_digest(records) -> tuple:
    a = np.asarray(list(records), dtype=np.int64).reshape(-1, 3)
    return a.shape[0], hashlib.blake2b(a.tobytes(), digest_size=16).hexdigest(), [tuple(r) for r in a[:8].tolist()]


class RecordedRecords:
    """(haystack, end_index, value) records the original produced, too many to keep: their count, a digest and the
    first few.  Equal to a record list with the same count and digest."""

    def __init__(self, n, digest, head):
        self.n, self.digest, self.head = n, digest, head

    def __eq__(self, other):
        return _records_digest(other)[:2] == (self.n, self.digest)

    def __repr__(self):
        return f"<{self.n} records of the original, blake2b {self.digest}, starting {self.head}>"


@pytest.fixture
def reference_records(request):
    """reference_records(label, compute) -> what compute(original bytes module) returned for this test, as recorded"""
    module, test = request.node.module.__name__, request.node.name

    def get(label, compute):
        if RECORDING is not None:
            import oracle
            n, digest, head = _records_digest(compute(oracle.ref_module("bytes")))
            RECORDING.setdefault(module, {})[f"{test}/{label}"] = (n, digest, head)
        else:
            got = load_traces(module).get(f"{test}/{label}")
            if got is None:
                pytest.fail(f"no recording of the original for {module}::{test}/{label} (tests/golden/record_reference.py)")
            n, digest, head = got
        return RecordedRecords(n, digest, head)
    return get


@pytest.fixture
def reference(request):
    """reference(flavour) -> the original extension of that flavour, as recorded for this test"""
    module = request.node.module.__name__
    test = request.node.name
    if RECORDING is not None:
        import oracle
        sessions = []

        def get(flavour):
            sessions.append((flavour, _Session()))
            return _Proxy(sessions[-1][1], oracle.ref_module(flavour), 0)
        yield get
        RECORDING.setdefault(module, {})[test] = [(fl, s.events) for fl, s in sessions]
        return
    traces = load_traces(module)
    if test not in traces:
        pytest.fail(f"no recording of the original for {module}::{test} (tests/golden/record_reference.py)")
    recorded = list(traces[test])
    sessions = []

    def get(flavour):
        if not recorded:
            pytest.fail(f"{test} asks for the original more often than it did when recorded")
        fl, events = recorded.pop(0)
        if fl != flavour:
            pytest.fail(f"{test} asks for the {flavour} original where the recording has the {fl} one")
        sessions.append(_Session(events))
        return _Proxy(sessions[-1], None, 0)
    failed = request.session.testsfailed
    yield get
    if request.session.testsfailed == failed:
        for s in sessions:
            assert s.pos == len(s.events), f"{test}: {len(s.events) - s.pos} recorded calls of the original never made"
