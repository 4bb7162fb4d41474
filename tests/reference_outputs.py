"""What the reference's own code returned, kept with the tests.

The test_oracle_ref_* modules hold the oracle to the reference's own C++, which oracle/Makefile (target `ref`) compiles into oracle/_ref/
only where the reference's sources are at hand.  So that those comparisons run on every machine, their `ref` fixture is a Reference: it
passes everything through to oracle.pyoracle except the ref_* calls, which answer from tests/golden/reference/<test module>.json.gz with
what the compiled reference returned for the same arguments.  An integer array of up to WHOLE_MAX_ITEMS values is stored whole; any other
array as a Fingerprint -- its dtype, shape and a hash of its bytes, one per field of a record array -- which assert_same checks as
np.testing.assert_array_equal would.

To record anew, build oracle/_ref (oracle/Makefile, target `ref`) and run the whole module with
CUBE_SLAM_RECORD_REFERENCE=1: the ref_* calls then run the compiled reference, the tests compare with its arrays directly, and the file
is rewritten when the module's tests are done.
"""
import gzip
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
RECORD = os.environ.get("CUBE_SLAM_RECORD_REFERENCE") == "1"
WHOLE_MAX_ITEMS = 512


def _hash_array(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a + 0)   # one NaN, and -0.0 as +0.0: assert_array_equal does not tell them apart either
    return hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()[:16]


def _feed(h, v):
    if isinstance(v, np.ndarray):
        h.update(("A%s%s" % (v.dtype.descr, v.shape)).encode() + np.ascontiguousarray(v).tobytes())
    elif hasattr(v, "_fields_"):                        # a ctypes parameter block: its fields, not its padding bytes
        _feed(h, [(f[0], getattr(v, f[0])) for f in v._fields_])
    elif isinstance(v, (list, tuple)):
        h.update(b"L%d" % len(v))
        for x in v:
            _feed(h, x)
    else:
        h.update(("S%s:%r" % (type(v).__name__, v)).encode())


def _call_key(name, args, kw):
    h = hashlib.sha256()
    _feed(h, [list(args), sorted(kw.items())])
    return "%s:%s" % (name, h.hexdigest()[:16])


class Fingerprint(object):
    """An array the reference returned, as its dtype, shape and the hash of its bytes ("<f4:271x4:<hash>" when stored)."""

    def __init__(self, s):
        dt, shape, self.sha = s.split(":")
        self.dtype, self.shape = np.dtype(dt), tuple(int(x) for x in shape.split("x") if x)

    @staticmethod
    def encode(a):
        return "%s:%s:%s" % (a.dtype.str, "x".join(map(str, a.shape)), _hash_array(a))

    def __len__(self):
        return self.shape[0]


class RecordFingerprint(object):
    """A record array the reference returned: its shape and one Fingerprint per field."""

    def __init__(self, d):
        self.shape = tuple(d["shape"])
        self.fields = {k: Fingerprint(v) for k, v in d["fields"].items()}

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, field):
        return self.fields[field]


def _encode(v):
    if isinstance(v, np.ndarray):
        if v.dtype.names:
            return {"shape": list(v.shape), "fields": {k: Fingerprint.encode(v[k]) for k in v.dtype.names}}
        if v.dtype.kind in "iu" and v.size <= WHOLE_MAX_ITEMS:
            return {"shape": list(v.shape), "dtype": v.dtype.str, "data": v.ravel().tolist()}
        return Fingerprint.encode(v)
    if isinstance(v, (list, tuple)):
        return [_encode(x) for x in v]
    return v.item() if isinstance(v, np.generic) else v


def _decode(v):
    if isinstance(v, list):
        return [_decode(x) for x in v]
    if isinstance(v, str):
        return Fingerprint(v)
    if not isinstance(v, dict):
        return v
    if "fields" in v:
        return RecordFingerprint(v)
    return np.array(v["data"], np.dtype(v["dtype"])).reshape(v["shape"])


def assert_same(got, want, err_msg=""):
    """np.testing.assert_array_equal(got, want) for a `want` the reference returned, stored whole or as a Fingerprint."""
    if not isinstance(want, Fingerprint):
        np.testing.assert_array_equal(got, want, err_msg=err_msg)
        return
    got = np.asarray(got)
    conv = got.astype(want.dtype)
    assert got.shape == want.shape, "%s: shape %s, the reference's %s" % (err_msg, got.shape, want.shape)
    assert np.array_equal(conv, got, equal_nan=got.dtype.kind in "fc"), "%s: %s values do not fit the reference's %s" % (err_msg, got.dtype, want.dtype)
    assert _hash_array(conv) == want.sha, "%s: differs from the reference's array (%s %s)" % (err_msg, want.dtype, want.shape)


class Reference(object):
    """oracle.pyoracle with its ref_* calls answered from the recording of one test module (see the module docstring)."""

    def __init__(self, oracle, module):
        self._oracle = oracle
        self._path = os.path.join(GOLD, module.rsplit(".", 1)[-1] + ".json.gz")
        if RECORD:
            self._calls = {}
        else:
            with gzip.open(self._path, "rt") as f:
                self._calls = json.load(f)

    def __getattr__(self, name):
        fn = getattr(self._oracle, name)
        if not name.startswith("ref_"):
            return fn

        def call(*args, **kw):
            key = _call_key(name, args, kw)
            if RECORD:
                out = fn(*args, **kw)
                self._calls[key] = _encode(out)
                return out
            assert key in self._calls, "%s: no recording of the reference for these arguments in %s" % (name, self._path)
            return _decode(self._calls[key])
        return call

    def save(self):
        """Write the recording (record mode only): one call per line, sorted, gzip without a time stamp."""
        if not RECORD:
            return
        text = "{\n" + ",\n".join("%s: %s" % (json.dumps(k), json.dumps(self._calls[k])) for k in sorted(self._calls)) + "\n}\n"
        os.makedirs(GOLD, exist_ok=True)
        with open(self._path, "wb") as f:
            f.write(gzip.compress(text.encode(), 9, mtime=0))
