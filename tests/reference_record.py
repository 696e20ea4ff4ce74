"""What the reference computed for a test, stored so that the comparison runs without it (tests/golden/reference_calls.json).

Where the reference is available (oracle/_ref built, or its shader tree present for the GLSL interpreter), a test calls it
live and every result is checked against the stored record; GLAVA_B200_RECORD_REFERENCE=1 rewrites the record instead.
Everywhere else the stored results are replayed in call order, each call's inputs checked by digest.  Arrays are stored
as digests: the comparisons that use them are bit for bit (same()), so a digest decides them exactly as the array would.
Arrays that a test compares within a tolerance are stored whole, compressed (call(..., whole=True))."""
import base64
import hashlib
import json
import os
import zlib

import numpy as np
import pytest

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json")
RECORD = os.environ.get("GLAVA_B200_RECORD_REFERENCE") == "1"

_store = None
_dirty = False


def _load():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(PATH):
            with open(PATH) as f:
                _store = json.load(f)
    return _store


def save():
    """called at the end of a recording session"""
    if _dirty:
        with open(PATH, "w") as f:
            json.dump(_load(), f, indent=0, sort_keys=True)
            f.write("\n")


def _digest(a, canonical_nan=False):
    a = np.ascontiguousarray(a)
    if canonical_nan and a.dtype.kind == "f":
        a = a.copy()
        a[np.isnan(a)] = np.nan
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:32]


class Recorded:
    """an array result of the reference known by its digests"""

    digest = staticmethod(_digest)

    def __init__(self, d):
        self.d = d


def same(ours, theirs, equal_nan=False):
    """ours equals the reference's result bit for bit (NaNs of any payload alike with equal_nan)"""
    ours = np.asarray(ours)
    if isinstance(theirs, Recorded):
        return _digest(ours, equal_nan) == theirs.d["nan" if equal_nan else "raw"]
    theirs = np.asarray(theirs)
    if equal_nan:
        return np.array_equal(ours, theirs, equal_nan=True)
    return ours.dtype == theirs.dtype and ours.shape == theirs.shape and ours.tobytes() == theirs.tobytes()


class Handle:
    """an opaque object the reference handed out (a channel), numbered in call order"""

    def __init__(self, index, obj=None):
        self.index, self.obj = index, obj


def _feed(h, a):
    """add one input to the digest h, independently of where the test runs: a file passed by its path as its name and
    contents, a directory as its files (the test's own, not entries linked in from elsewhere), an absolute path that does
    not exist as its name"""
    if isinstance(a, np.ndarray):
        h.update(b"a" + _digest(a).encode())
    elif isinstance(a, Handle):
        h.update(b"h%d" % a.index)
    elif a is None:
        h.update(b"N")
    elif isinstance(a, (bool, int, float, np.floating, np.integer)):
        h.update(b"n" + repr(float(a)).encode())
    elif hasattr(a, "_fields_"):
        h.update(b"s" + bytes(a))
    elif isinstance(a, str) and os.path.isfile(a):
        with open(a, "rb") as f:
            h.update(b"f" + os.path.basename(a).encode() + b"\0" + f.read())
    elif isinstance(a, str) and os.path.isdir(a):
        h.update(b"d")
        for name in sorted(os.listdir(a)):
            path = os.path.join(a, name)
            if not os.path.islink(path):
                _feed(h, path)
    elif isinstance(a, str) and os.path.isabs(a):
        h.update(b"m" + os.path.basename(a).encode())
    elif isinstance(a, str):
        h.update(b"t" + a.encode())
    elif isinstance(a, (list, tuple)):
        h.update(b"[%d" % len(a))
        for v in a:
            _feed(h, v)
    elif isinstance(a, dict):
        h.update(b"{%d" % len(a))
        for k in sorted(a):
            _feed(h, k); _feed(h, a[k])
    else:
        raise TypeError(f"no digest for an input of type {type(a).__name__}")


def _in_digest(args, kw):
    """digest of a call's inputs (_feed)"""
    h = hashlib.sha256()
    for a in list(args) + [kw[k] for k in sorted(kw)]:
        _feed(h, a)
    return h.hexdigest()[:32]


def _encode(out):
    if isinstance(out, np.ndarray):
        return {"array": {"raw": _digest(out), "nan": _digest(out, True)}}
    if isinstance(out, tuple):
        out = list(out)
    return {"value": out}


def _decode(rec):
    if "array" in rec:
        return Recorded(rec["array"])
    if "raises" in rec:
        raise ValueError("the reference rejected its input (recorded)")
    return rec["value"]


class Session:
    """the calls of one test: recorded, checked against the record, or replayed"""

    def __init__(self, request, live):
        self.key = os.path.basename(request.node.fspath) + "::" + request.node.name
        self.live = live
        stored = _load().get(self.key)
        if RECORD and live:
            self.calls, self.stored = [], None
        elif stored is None:
            pytest.fail(f"no recorded reference results for {self.key}: run it once with the reference built and "
                        "GLAVA_B200_RECORD_REFERENCE=1")
        else:
            self.calls, self.stored = None, stored
        self.pos = 0
        request.addfinalizer(self.finish)

    def _next(self, name, din):
        assert self.pos < len(self.stored), f"{self.key}: more reference calls than recorded"
        rec = self.stored[self.pos]
        self.pos += 1
        assert (rec["call"], rec["in"]) == (name, din), f"{self.key}: call {self.pos} is {name} on other inputs than recorded"
        return rec

    def call(self, name, fn, args=(), kw=None, whole=False, handle=False, check_live=True):
        """fn(*args, **kw) through the record; whole: store an array result as its values, not its digest; handle: the
        result is an opaque object, only the call itself is recorded; check_live=False: a live result need not equal the
        recorded one (it may hold memory the reference never initialised; the test compares only what it defines)"""
        kw = kw or {}
        din = _in_digest(args, kw)
        if handle:
            if self.live:
                out = fn(*args, **kw)
                rec = {"call": name, "in": din, "value": None}
                if self.calls is not None:
                    self.calls.append(rec)
                else:
                    assert self._next(name, din) == rec
                return out
            self._next(name, din)
            return None
        if not self.live:
            rec = self._next(name, din)
            out = rec.get("whole")
            if out is not None:
                raw = zlib.decompress(base64.b64decode(out["zb64"]))
                return np.frombuffer(raw, dtype=out["dtype"]).reshape(out["shape"]).copy()
            return _decode(rec)
        try:
            out = fn(*args, **kw)
            rec = {"call": name, "in": din}
            if whole:
                a = np.ascontiguousarray(out)
                rec["whole"] = {"dtype": a.dtype.str, "shape": list(a.shape), "zb64": base64.b64encode(zlib.compress(a.tobytes(), 9)).decode()}
            else:
                rec.update(_encode(out))
        except ValueError as e:
            rec = {"call": name, "in": din, "raises": "ValueError"}
            out = e
        if self.calls is not None:
            self.calls.append(rec)
        elif check_live:
            assert self._next(name, din) == rec, f"{self.key}: the reference's result of call {self.pos} ({name}) is not the recorded one"
        else:
            self._next(name, din)
        if isinstance(out, ValueError):
            raise out
        return out

    def finish(self):
        global _dirty
        if self.calls is not None:
            _load()[self.key] = self.calls
            _dirty = True
        else:
            assert self.pos == len(self.stored), f"{self.key}: {len(self.stored) - self.pos} recorded reference calls not made"


class ReferenceProxy:
    """oracle.oracle.Reference through a Session: same methods; chan() returns a Handle"""

    def __init__(self, session, live_ref):
        self._s, self._ref, self._chans = session, live_ref, 0

    def chan(self, p):
        """a channel with the transform parameters of p; the parameters are part of the record"""
        h = Handle(self._chans)
        self._chans += 1
        h.obj = self._s.call("chan", lambda q: self._ref.chan(q) if self._ref else None, (p,), handle=True)
        return h

    def __getattr__(self, name):
        fn = getattr(self._ref, name) if self._ref else None

        def call(*args, **kw):
            live = lambda *a, **k: fn(*[x.obj if isinstance(x, Handle) else x for x in a], **k)   # noqa: E731
            return self._s.call(name, live, args, kw)
        return call
