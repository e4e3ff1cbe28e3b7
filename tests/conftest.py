import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "hotpath_v1.npz"))


@pytest.fixture(scope="session")
def blosum():
    import numpy as np
    d = np.load(os.path.join(ROOT, "tests", "golden", "blosum62.npz"))
    return d["mat"], d["pback"]


@pytest.fixture(scope="session")
def oracle(blosum):
    from oracle.pyoracle import Oracle, build
    build(with_ref=False)
    return Oracle(*blosum)


REF_CALLS = os.path.join(ROOT, "tests", "golden", "ref_calls_v1.pkl.xz")
DB_SUFFIXES = ("", ".index", ".dbtype")


def _fingerprint(x, h):
    """hash of a call's arguments; of a path only the file name counts (tests write under a fresh tmp_path)"""
    import numpy as np
    if isinstance(x, (np.ndarray, np.generic)):
        x = np.ascontiguousarray(x)
        h.update(("a%s%s" % (x.dtype.str, x.shape)).encode())
        h.update(x.tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d" % len(x))
        for y in x:
            _fingerprint(y, h)
    elif isinstance(x, dict):
        for k in sorted(x):
            _fingerprint(k, h)
            _fingerprint(x[k], h)
    elif isinstance(x, (bytes, bytearray)):
        h.update(b"b%d" % len(x))
        h.update(bytes(x))
    elif isinstance(x, str):
        h.update(("s" + (os.path.basename(x) if os.sep in x else x)).encode())
    else:
        h.update(("r" + repr(x)).encode())


def _call_id(name, args, kwargs):
    import hashlib
    h = hashlib.sha1(name.encode())
    _fingerprint([list(args), kwargs], h)
    return h.digest()[:4]


class _RecordingRef:
    """Forwards to the reference's own code (oracle/_ref) and keeps every answer, and the files db_write leaves, in call order."""

    def __init__(self, calls):
        from oracle.pyoracle import Ref
        self._ref, self._calls = Ref(), calls

    def __getattr__(self, name):
        import pickle

        def call(*args, **kwargs):
            out = getattr(self._ref, name)(*args, **kwargs)
            files = [open(args[0] + s, "rb").read() for s in DB_SUFFIXES] if name == "db_write" else None
            self._calls.append((name, _call_id(name, args, kwargs), pickle.dumps((out, files), protocol=4)))
            return out
        return call


class _ReplayedRef:
    """Answers the calls a test makes to the reference with what the reference answered when the recording was made; a call
    with other arguments than then is an error, not a stale answer."""

    def __init__(self, calls, test):
        self._calls, self._test, self._next = calls, test, 0

    def __getattr__(self, name):
        import pickle

        def call(*args, **kwargs):
            if self._next >= len(self._calls):
                raise AssertionError("%s: call %d (%s) is not in %s" % (self._test, self._next, name, REF_CALLS))
            rec_name, rec_id, blob = self._calls[self._next]
            if (rec_name, rec_id) != (name, _call_id(name, args, kwargs)):
                raise AssertionError("%s: call %d is %s with other inputs than the recorded %s; re-record with B200_RECORD_REF=1"
                                     % (self._test, self._next, name, rec_name))
            self._next += 1
            out, files = pickle.loads(blob)
            for s, data in zip(DB_SUFFIXES, files or ()):
                with open(args[0] + s, "wb") as f:
                    f.write(data)
            return out
        return call


@pytest.fixture(scope="session")
def _ref_calls():
    import lzma
    import pickle
    stored, recorded = {}, {}
    if os.path.exists(REF_CALLS):
        with lzma.open(REF_CALLS, "rb") as f:
            stored = pickle.load(f)
    yield stored, recorded
    if recorded:
        stored.update(recorded)
        with lzma.open(REF_CALLS, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
            pickle.dump(stored, f, protocol=4)


@pytest.fixture
def ref(request, _ref_calls):
    """The reference's own hot-path code (oracle.pyoracle.Ref), answered from tests/golden/ref_calls_v1.pkl.xz.  With
    B200_RECORD_REF=1 (and oracle/_ref built) the live reference answers instead and the recording of this test is replaced."""
    stored, recorded = _ref_calls
    test = request.node.nodeid.split("/")[-1]
    if os.environ.get("B200_RECORD_REF") == "1":
        recorded[test] = []
        yield _RecordingRef(recorded[test])
        return
    if test not in stored:
        raise AssertionError("no recorded reference calls for %s in %s" % (test, REF_CALLS))
    replay = _ReplayedRef(stored[test], test)
    yield replay
    assert replay._next == len(stored[test]), "%s made %d of its %d recorded reference calls" % (test, replay._next, len(stored[test]))


@pytest.fixture(scope="session")
def built_lib():
    from mmseqs2_b200 import build as b
    return b.build()


@pytest.fixture(scope="session")
def submat(blosum, built_lib):
    from mmseqs2_b200 import SubMatrix
    return SubMatrix(*blosum)


@pytest.fixture(scope="session")
def ctx(built_lib):
    from mmseqs2_b200 import Context
    c = Context(0)
    yield c
    c.close()
