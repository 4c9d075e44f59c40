"""The compiled reference's answers, recorded for the tests (not product code).

The parity tests call the unmodified reference through oracle.binding.RefShim, which needs oracle/_ref (built only
where the reference sources are).  Every call a test makes is recorded once, with a digest of its arguments, under
tests/golden/ref/<test module>/<test>.npz.xz; elsewhere the tests replay those answers in the same order, and a call
whose arguments differ from the recorded ones fails the test instead of answering it.  The comparisons in the tests
are the same either way.  Of a result dict only the entries the test read are stored.  A test whose answers do not
fit in MAX_FILE_BYTES is not recorded and needs oracle/_ref.  The sequence weights of the alignment reader go through
the host's RCPPS reciprocal estimate, whose bits differ between CPU vendors; the stored answers are an Intel host's.

    HHG_REF_RECORD=<dir> python -m pytest tests ...     (needs oracle/_ref; writes <dir>/<test module>/<test>.npz.xz)
"""
from __future__ import annotations

import glob
import hashlib
import io
import json
import lzma
import os
import re

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
# a test with an answer larger than MAX_RESULT_BYTES (crf_text: 7 MB) or a recording larger than MAX_FILE_BYTES
# (compressed) is not recorded; it needs oracle/_ref
MAX_RESULT_BYTES = 4 << 20
MAX_FILE_BYTES = 900 << 10


def _path(root, key):
    """<root>/<test module>/<test name with parameters>.npz.xz for the key '<module file>::<test name>'."""
    mod, name = key.split("::", 1)
    return os.path.join(root, os.path.splitext(mod)[0], re.sub(r"[^\w.\-\[\]]", "_", name) + ".npz.xz")


def _feed(h, x):
    """Canonical bytes of a call argument; file paths (and path prefixes of ffindex triples) by their contents."""
    if x is None or isinstance(x, (bool, int, float)):
        h.update(repr(x).encode())
    elif isinstance(x, str):
        files = [x] if os.path.isfile(x) else sorted(glob.glob(x + "*")) if os.sep in x else []
        if files:
            for f in files:
                h.update(b"file" + os.path.basename(f)[len(os.path.basename(x)):].encode())
                with open(f, "rb") as fh:
                    h.update(fh.read())
        else:
            h.update(b"str" + x.encode())
    elif isinstance(x, bytes):
        h.update(b"bytes" + x)
    elif isinstance(x, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(x)
        h.update(f"nd{a.dtype.str}{a.shape}".encode() + a.tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(f"seq{len(x)}".encode())
        for v in x:
            _feed(h, v)
    elif isinstance(x, dict):
        for k in sorted(x):
            h.update(f"key{k}".encode())
            _feed(h, x[k])
    else:
        raise TypeError(f"cannot digest a {type(x).__name__} argument")


def digest(name, args, kwargs):
    h = hashlib.sha256(name.encode())
    _feed(h, list(args))
    _feed(h, kwargs)
    return h.hexdigest()[:24]


class _Tracked(dict):
    """A result dict that notes which entries the test read."""

    def __init__(self, *a):
        super().__init__(*a)
        self.used = set()

    def __getitem__(self, k):
        self.used.add(k)
        return super().__getitem__(k)

    def get(self, k, default=None):
        self.used.add(k)
        return super().get(k, default)

    def _all(self, fn):
        self.used.update(super().keys())
        return fn()

    def keys(self):
        return self._all(super().keys)

    def values(self):
        return self._all(super().values)

    def items(self):
        return self._all(super().items)

    def __iter__(self):
        return self._all(super().__iter__)

    def copy(self):
        return self._all(lambda: dict(super(_Tracked, self).items()))


def _track(x):
    if isinstance(x, dict):
        return _Tracked({k: _track(v) for k, v in x.items()})
    if isinstance(x, (list, tuple)):
        return type(x)(_track(v) for v in x)
    return x


def _enc(x, put):
    """JSON-able form of a result; put(array) stores an array and returns its number."""
    from oracle.binding import PrepParams
    if x is None or isinstance(x, (bool, int, float, str)):
        return {"v": x}
    if isinstance(x, (np.ndarray, np.generic, bytes)):
        k = put(np.frombuffer(x, np.uint8) if isinstance(x, bytes) else np.asarray(x))
        return {"b" if isinstance(x, bytes) else "s" if isinstance(x, np.generic) else "a": k}
    if isinstance(x, PrepParams):
        return {"pp": [getattr(x, f) for f, _ in x._fields_]}
    if isinstance(x, _Tracked):
        return {"d": [[k, _enc(dict.__getitem__(x, k), put)] for k in dict.keys(x) if k in x.used]}
    if isinstance(x, dict):
        return {"d": [[k, _enc(v, put)] for k, v in x.items()]}
    if isinstance(x, (list, tuple)):
        return {"l" if isinstance(x, list) else "t": [_enc(v, put) for v in x]}
    raise TypeError(f"cannot record a {type(x).__name__} result")


def _dec(e, arrays):
    from oracle.binding import PrepParams
    (tag, v), = e.items()
    if tag == "v":
        return v
    if tag == "a":
        return arrays[v].copy()
    if tag == "s":
        return arrays[v][()]
    if tag == "b":
        return arrays[v].tobytes()
    if tag == "pp":
        return PrepParams(*v)
    if tag == "d":
        return {k: _dec(x, arrays) for k, x in v}
    return [_dec(x, arrays) for x in v] if tag == "l" else tuple(_dec(x, arrays) for x in v)


def _nbytes(x):
    if isinstance(x, (np.ndarray, bytes)):
        return len(x) if isinstance(x, bytes) else x.nbytes
    if isinstance(x, dict):
        return sum(_nbytes(v) for v in dict.values(x))
    if isinstance(x, (list, tuple)):
        return sum(_nbytes(v) for v in x)
    return 8


def load(key):
    """(attributes, [(method, digest, encoded result)]) and the arrays of one test's recording, or None."""
    path = _path(GOLD, key)
    if not os.path.exists(path):
        return None
    with open(path, "rb") as f:
        z = np.load(io.BytesIO(lzma.decompress(f.read())))
    n = sum(1 for k in z.files if k.startswith("a"))
    return json.loads(z["index"].tobytes()), [z[f"a{k}"] for k in range(n)]


class Recorder:
    """The live RefShim, with every public call of one test appended to `calls` (None once a call was too large)."""

    def __init__(self, live, sink):
        self._live, self._sink = live, sink
        self.V = live.V

    def __getattr__(self, name):
        fn = getattr(self._live, name)
        if name.startswith("_") or not callable(fn):
            return fn

        def call(*args, **kwargs):
            d = digest(name, args, kwargs)
            r = _track(fn(*args, **kwargs))
            if self._sink["calls"] is not None:
                if _nbytes(r) > MAX_RESULT_BYTES:
                    self._sink["calls"] = None
                else:
                    self._sink["calls"].append((name, d, r))
            return r
        return call


class Replayer:
    """Answers one test's calls from its recording, in order, checking each call's arguments against the recorded ones."""

    def __init__(self, nodeid, entry, arrays):
        attrs, self._calls = entry
        self._nodeid, self._arrays, self._next = nodeid, arrays, 0
        self.V = attrs["V"]

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def call(*args, **kwargs):
            k = self._next
            assert k < len(self._calls), f"{self._nodeid}: call {k} ({name}) was not recorded"
            rname, rdig, res = self._calls[k]
            assert rname == name and rdig == digest(name, args, kwargs), \
                f"{self._nodeid}: call {k} {name} differs from the recorded call {rname} (inputs changed: record again)"
            self._next += 1
            return _dec(res, self._arrays)
        return call


def save(key, V, calls, out_dir):
    """Write one test's recording under out_dir (identical arrays stored once); False when it is too large."""
    arrays, seen = [], {}

    def put(a):
        a = np.ascontiguousarray(a)
        h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest()
        if h not in seen:
            seen[h] = len(arrays)
            arrays.append(a)
        return seen[h]
    index = [{"V": V}, [(n, d, _enc(r, put)) for n, d, r in calls]]
    buf = io.BytesIO()
    np.savez(buf, index=np.frombuffer(json.dumps(index).encode(), np.uint8), **{f"a{k}": a for k, a in enumerate(arrays)})
    data = lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME)
    if len(data) > MAX_FILE_BYTES:
        return False
    path = _path(out_dir, key)
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "wb") as f:
        f.write(data)
    return True
