"""Shared test helpers: one parameter dict feeds both the oracle (checker) and the product."""
import numpy as np

from oracle import oracle as O
from semantic_suma_b200 import api, synth
from reference_replay import Recorded, array_digest

_cache = {}


def both_params(**kw):
    return O.default_params(**kw), api.default_params(**kw)


def sized(width, height=64, **kw):
    d = dict(data_width=width, model_width=width, data_height=height, model_height=height)
    d.update(kw)
    return d


def scans(width, height=64, n=3, semantic=False, **kw):
    key = (width, height, n, semantic, tuple(sorted(kw.items())))
    if key not in _cache:
        sc = synth.Scene(width=width, height=height, semantic=semantic, **kw)
        poses = synth.trajectory(n)
        _cache[key] = ([sc.scan(f, poses[f]) for f in range(n)], poses)
    return _cache[key]


def bits(a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        v = a.view(np.uint32).copy()
        v[np.isnan(a)] = 0x7fc00000  # all NaNs compare equal (x86 and sm_100a use different default payloads)
        return v
    if a.dtype == np.float64:
        v = a.view(np.uint64).copy()
        v[np.isnan(a)] = 0x7ff8000000000000
        return v
    return a


def assert_bits_equal(a, b, what=""):
    if isinstance(a, Recorded) or isinstance(b, Recorded):  # a replayed output of the reference: compare digests
        assert tuple(np.shape(a) if not isinstance(a, Recorded) else a.shape) == \
            tuple(np.shape(b) if not isinstance(b, Recorded) else b.shape), "%s: shape differs" % what
        da, db = array_digest(a), array_digest(b)
        assert da == db, "%s: differs from the reference's output (digest %s vs %s)" % (what, da, db)
        return
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    ba, bb = bits(a), bits(b)
    bad = np.argwhere(ba != bb)
    if bad.size:
        i = tuple(bad[0])
        raise AssertionError("%s: %d / %d elements differ; first at %s: %r vs %r" %
                             (what, bad.shape[0], ba.size, i, a[i], b[i]))


def surfel_fields_equal(a, b, what="surfels"):
    assert a.shape == b.shape, "%s: count %d vs %d" % (what, a.shape[0], b.shape[0])
    if isinstance(a, Recorded) or isinstance(b, Recorded):  # a replayed output of the reference: one digest, all fields
        return assert_bits_equal(a, b, what)
    for f in a.dtype.names:
        assert_bits_equal(a[f], b[f], "%s.%s" % (what, f))
