"""The reference's outputs that the tests compare with, replayed from tests/golden/reference_calls/<test module>.json.

Every call a test makes on oracle/ref.py (the reference's own sources and shaders, compiled from a checkout of the
reference into oracle/_ref/) is recorded once, in call order per test, and replayed on every later run, so that the
comparisons need neither the reference nor oracle/_ref. A recorded value keeps small arrays and scalars whole; an array
of more than SMALL elements (or any array, inside `with R.digests():`) keeps its shape, dtype and digest, which is all
a bit-for-bit comparison needs. Inside `with R.sampled(part):` that part of the call's output also keeps the digest of
each image channel and the values of a fixed, seeded sample of SAMPLE pixels, for the comparisons made within
tolerances (R.sample).

Each record also holds a digest of the call's array and number arguments: a replayed output is only used for the
inputs it was recorded with.

    SUMA_RECORD_REFERENCE=1 python -m pytest tests/test_ref_shaders.py tests/test_ref_full.py tests/test_ref_host.py
    SUMA_RECORD_REFERENCE=1 python -m pytest tests/test_gpu_parity.py -m gpu --cusim -k reference_shaders_directly
(re-records; needs oracle/_ref built from the reference)
"""
import atexit
import base64
import ctypes
import hashlib
import json
import os
from contextlib import contextmanager

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls")
RECORD = os.environ.get("SUMA_RECORD_REFERENCE") == "1"
SMALL = 4096
SAMPLE = 512


def _canonical(a):
    """bytes of an array with every NaN in one canonical encoding (x86 and sm_100a use different default payloads)"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f" and a.dtype.itemsize in (4, 8):
        v = a.view(np.uint32 if a.dtype.itemsize == 4 else np.uint64).copy()
        v[np.isnan(a)] = 0x7fc00000 if a.dtype.itemsize == 4 else 0x7ff8000000000000
        a = v
    return a.tobytes()


def _h(*parts):
    h = hashlib.sha256()
    for p in parts:
        h.update(p if isinstance(p, bytes) else str(p).encode())
    return h.hexdigest()[:16]


def array_digest(a):
    if isinstance(a, Recorded):
        return a.digest
    a = np.asarray(a)
    if a.dtype.names:
        return _h(a.shape, *[array_digest(a[f]) for f in a.dtype.names])
    return _h(a.dtype.str, a.shape, _canonical(a))


class Recorded:
    """a large array of the reference, replayed: shape, dtype and digest, plus channel digests and a pixel sample where
    they were recorded"""

    def __init__(self, rec):
        self.shape, self.dtype, self.digest = tuple(rec["shape"]), np.dtype(rec["dtype"]), rec["digest"]
        self._channels, self._sample = rec.get("channels"), rec.get("sample")

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, key):
        if isinstance(key, tuple) and len(key) == 2 and key[0] is Ellipsis and self._channels:
            return Recorded({"shape": self.shape[:-1], "dtype": self.dtype.str,
                             "digest": self._channels[key[1] % self.shape[-1]]})
        raise TypeError("a replayed output of the reference supports channel selection only, and only where recorded")

    def __repr__(self):
        return "<reference output %s %s %s>" % (self.dtype, self.shape, self.digest)


def _sample_index(shape):
    pixels = int(np.prod(shape[:-1])) if len(shape) > 1 else int(shape[0])
    return np.sort(np.random.default_rng(0).choice(pixels, min(SAMPLE, pixels), replace=False))


def sample(x):
    """(pixel indices, values at them) of an output recorded inside `with R.sampled(...)` (or of a live array)"""
    idx = _sample_index(x.shape)
    if isinstance(x, Recorded):
        return idx, _decode(x._sample)
    x = np.asarray(x)
    return idx, (x.reshape(-1, x.shape[-1]) if x.ndim > 1 else x)[idx]


def _encode_array(a, with_sample):
    if not _store.digests and a.size <= SMALL and not a.dtype.names:
        return {"array": base64.b64encode(np.ascontiguousarray(a).tobytes()).decode(), "dtype": a.dtype.str,
                "shape": list(a.shape)}
    rec = {"shape": list(a.shape), "dtype": a.dtype.str, "digest": array_digest(a)}
    if with_sample:
        rec["channels"] = [array_digest(a[..., c]) for c in range(a.shape[-1])]
        rec["sample"] = _encode(sample(a)[1])
    return rec


def _encode(v, part=None):
    """part: the element of a tuple (True: the value itself) that also keeps channel digests and a pixel sample"""
    if isinstance(v, np.ndarray):
        return {"nd": _encode_array(v, part is True)}
    if isinstance(v, np.generic):
        return {"nd": _encode_array(np.asarray(v), False), "scalar": True}
    if isinstance(v, tuple):
        return {"tuple": [_encode(x, True if i == part else None) for i, x in enumerate(v)]}
    if isinstance(v, list):
        return [_encode(x) for x in v]
    if isinstance(v, dict):
        return {"dict": {k: _encode(x) for k, x in v.items()}}
    assert v is None or isinstance(v, (bool, int, float, str)), type(v)
    return v


def _decode(v):
    if isinstance(v, list):
        return [_decode(x) for x in v]
    if not isinstance(v, dict):
        return v
    if "tuple" in v:
        return tuple(_decode(x) for x in v["tuple"])
    if "dict" in v:
        return {k: _decode(x) for k, x in v["dict"].items()}
    rec = v["nd"]
    if "array" not in rec:
        return Recorded(rec)
    a = np.frombuffer(base64.b64decode(rec["array"]), np.dtype(rec["dtype"])).reshape(rec["shape"]).copy()
    return a[()] if v.get("scalar") else a


def _args_digest(args, kwargs):
    """what the call computed from: arrays, numbers, names and parameter blocks (not paths, which differ between runs)"""
    parts = []

    def walk(x):
        if isinstance(x, (np.ndarray, Recorded)):
            parts.append(array_digest(x))
        elif isinstance(x, ctypes.Structure):
            parts.append(_h(bytes(x)))
        elif isinstance(x, (list, tuple)):
            for y in x:
                walk(y)
        elif isinstance(x, (bool, int, float, np.generic)):
            parts.append(repr(float(x)))
        elif isinstance(x, str) and os.sep not in x:
            parts.append(x)
    walk(list(args))
    walk([kwargs[k] for k in sorted(kwargs)])
    return _h(*parts)[:8]


def _current_test():
    cur = os.environ.get("PYTEST_CURRENT_TEST", "")
    path, _, name = cur.rsplit(" ", 1)[0].partition("::")
    assert name, "the reference's outputs are replayed inside a test only"
    return os.path.splitext(os.path.basename(path))[0], name


class _Store:
    def __init__(self):
        self.files, self.counters, self.recorded, self.sampling, self.paused = {}, {}, set(), None, False
        self.digests = False

    def _records(self, module):
        if module not in self.files:
            path = os.path.join(GOLDEN, module + ".json")
            self.files[module] = json.load(open(path)) if os.path.exists(path) else {}
        return self.files[module]

    def call(self, what, fn, args, kwargs):
        module, test = _current_test()
        key = (module, test)
        i = self.counters.get(key, 0)
        self.counters[key] = i + 1
        recs = self._records(module)
        dig = _args_digest(args, kwargs)
        if RECORD:
            if key not in self.recorded:
                recs[test] = []
                self.recorded.add(key)
            self.paused = True
            try:
                out = fn()
            finally:
                self.paused = False
            recs[test].append([what, dig, _encode(out, self.sampling)])
            return out
        assert test in recs and i < len(recs[test]), \
            "%s::%s: no recorded output of the reference for call %d (%s)" % (module, test, i, what)
        call, args, out = recs[test][i]
        assert (call, args) == (what, dig), \
            "%s::%s call %d: %s on inputs %s, recorded: %s on inputs %s" % (module, test, i, what, dig, call, args)
        return _decode(out)

    def save(self):
        for module in {m for m, _ in self.recorded}:
            os.makedirs(GOLDEN, exist_ok=True)
            recs = self.files[module]
            with open(os.path.join(GOLDEN, module + ".json"), "w") as f:  # one line per call
                f.write("{\n" + ",\n".join("%s: [\n%s\n]" % (json.dumps(t), ",\n".join(
                    json.dumps(r, separators=(",", ":"), sort_keys=True) for r in recs[t])) for t in sorted(recs)) + "\n}\n")


_store = _Store()
if RECORD:
    atexit.register(_store.save)


def _ref():
    from oracle import ref
    return ref


class _Object:
    """an object of oracle/ref.py (Map, Full): constructed and called live while recording, replayed otherwise"""

    def __init__(self, cls, args, kwargs):
        self._cls, self._obj = cls, None

        def make():
            self._obj = getattr(_ref(), cls)(*args, **kwargs)
        _store.call(cls, make, args, kwargs)

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def method(*args, **kwargs):
            if _store.paused:
                return getattr(self._obj, name)(*args, **kwargs)
            return _store.call("%s.%s" % (self._cls, name), lambda: getattr(self._obj, name)(*args, **kwargs), args, kwargs)
        return method


class _Reference:
    """stands in for `from oracle import ref as R` in the tests"""

    @staticmethod
    @contextmanager
    def sampled(part):
        """the calls inside keep channel digests and a pixel sample of output[part]"""
        _store.sampling = part
        try:
            yield
        finally:
            _store.sampling = None

    sample = staticmethod(sample)

    @staticmethod
    @contextmanager
    def digests():
        """the calls inside keep only digests, also of small arrays (outputs compared bit for bit)"""
        _store.digests = True
        try:
            yield
        finally:
            _store.digests = False

    @staticmethod
    def computed(fn):
        """a value the test derives from the reference's outputs alone (fn runs on the live reference while recording)"""
        return _store.call("computed", fn, (), {})

    def Map(self, *args, **kwargs):
        return self._object("Map", args, kwargs)

    def Full(self, *args, **kwargs):
        return self._object("Full", args, kwargs)

    @staticmethod
    def _object(cls, args, kwargs):
        if _store.paused:
            return getattr(_ref(), cls)(*args, **kwargs)
        return _Object(cls, args, kwargs)

    def __getattr__(self, name):
        def fn(*args, **kwargs):
            if _store.paused:
                return getattr(_ref(), name)(*args, **kwargs)
            return _store.call(name, lambda: getattr(_ref(), name)(*args, **kwargs), args, kwargs)
        return fn


R = _Reference()
