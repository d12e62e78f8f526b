"""pytest configuration: the `gpu` marker and shared fixtures.

`-m "not gpu"` runs on a CPU-only host: oracle vs reference vs golden vectors, host
logic, C-ABI symbol checks.  `-m gpu` are the parity tests proper: they call the CUDA
engine through its C-ABI and compare against the oracle.
"""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _has_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device on this host")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class PinnedOracle:
    """The restatement (oracle/adb_oracle.c) with the unmodified reference objects (oracle/_ref)
    run beside it: for the operators the reference computes without reading out of bounds,
    every call is made on BOTH and the answers must be identical before the restatement's is
    returned.  GPU parity tests that take `port` are thereby checked against the reference
    itself wherever oracle/_ref exists (this container; on the GPU box the prebuilt objects
    travel with the snapshot)."""
    SAFE = ("select_scan", "select_result", "fetch", "sum", "add", "sub", "chain_select_fetch_sum")

    def __init__(self, port, ref):
        self._port, self._ref = port, ref

    def __getattr__(self, name):
        fn = getattr(self._port, name)
        if self._ref is None or name not in self.SAFE:
            return fn
        rfn = getattr(self._ref, name)

        def both(*a, **kw):
            x, y = fn(*a, **kw), rfn(*a, **kw)
            same = np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y
            assert same, f"oracle restatement and reference disagree on {name}"
            return x
        return both


REFERENCE_ANSWERS = os.path.join(ROOT, "tests", "golden", "reference_answers.json")


def digest(x) -> str:
    """128-bit digest of a call's arguments or answer: arrays by dtype, shape and bytes; ints,
    floats (nan included), bools, None, bytes and tuples / lists of those by value."""
    h = hashlib.sha256()

    def feed(v):
        if isinstance(v, np.ndarray):
            a = np.ascontiguousarray(v)
            h.update(b"a%s%s:" % (a.dtype.str.encode(), repr(a.shape).encode()))
            h.update(a.tobytes())
        elif isinstance(v, (tuple, list)):
            h.update(b"(%d" % len(v))
            for e in v:
                feed(e)
            h.update(b")")
        elif v is None:
            h.update(b"n")
        elif isinstance(v, (bool, np.bool_)):
            h.update(b"b%d" % bool(v))
        elif isinstance(v, (int, np.integer)):
            h.update(b"i%d" % int(v))
        elif isinstance(v, (float, np.floating)):
            h.update(b"f" + float(v).hex().encode())
        elif isinstance(v, bytes):
            h.update(b"y%d:" % len(v) + v)
        elif isinstance(v, str):
            feed(v.encode())
        else:
            raise TypeError(f"cannot digest {type(v).__name__}")
    feed(x)
    return h.hexdigest()[:32]


class RecordedReference:
    """The reference operators (oracle/_ref) as recorded in tests/golden/reference_answers.json:
    for every call the tests make on them, a digest of the arguments maps to a digest of the
    reference's answer.  Where oracle/_ref is not built, a call is answered by the restatement,
    and that answer must have the recorded reference answer's digest -- so a test that compares
    with the reference still does, bit for bit, on the inputs it was recorded with.

    ADB_RECORD_REFERENCE=<file> records instead: the answers of oracle/_ref when it is built,
    else of the restatement, are merged into <file> at the end of the session (the restatement's
    answers were recorded at a commit where they equalled oracle/_ref's on every one of these
    calls).  Copy the file over tests/golden/reference_answers.json to keep it."""

    def __init__(self, impl, opt: str, answers: dict, recording: bool):
        self._impl, self._opt, self._answers, self._recording = impl, opt, answers, recording

    def __getattr__(self, name):
        fn = getattr(self._impl, name)

        def call(*a, **kw):
            out = fn(*a, **kw)
            key, got = digest((self._opt, name, a, sorted(kw.items()))), digest(out)
            if self._recording:
                assert self._answers.setdefault(key, got) == got, f"two answers recorded for one {name} call"
            else:
                want = self._answers.get(key)
                assert want is not None, (f"no recorded reference answer for this {name} call: record one "
                                          "with ADB_RECORD_REFERENCE where oracle/_ref is built")
                assert got == want, f"the restatement's {name} differs from the reference's recorded answer"
            return out
        return call


@pytest.fixture(scope="session")
def _reference_answers():
    record = os.environ.get("ADB_RECORD_REFERENCE")
    answers = {}
    if os.path.exists(record or REFERENCE_ANSWERS):
        with open(record or REFERENCE_ANSWERS) as f:
            answers = json.load(f)
    yield answers, bool(record)
    if record:
        with open(record, "w") as f:
            json.dump(dict(sorted(answers.items())), f, indent=0)
            f.write("\n")


def _reference(opt, answers):
    from oracle import oracle
    answers, recording = answers
    r = oracle.reference(opt)
    if r is not None and not recording:
        return r
    return RecordedReference(r or oracle.port(), opt, answers, recording)


@pytest.fixture(scope="session")
def port():
    from oracle import oracle
    return PinnedOracle(oracle.port(), oracle.reference("O2"))


@pytest.fixture(scope="session")
def ref(_reference_answers):
    return _reference("O2", _reference_answers)


@pytest.fixture(scope="session")
def ref_o0(_reference_answers):
    return _reference("O0", _reference_answers)


@pytest.fixture
def rng():
    return np.random.default_rng(42)
