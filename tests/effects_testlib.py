"""Recorded reference results of the image-effect tests (test_effects_cpu.py, test_gpu_effects.py).

Same scheme as uhdr_testlib.from_reference / reference_file: where the reference build (oracle/_ref) is present it
computes the answer, everywhere else the SHA-256 recorded from it stands in.  The effect keys ("effects/...") are kept
in their own file, tests/golden/effects_reference_digests.json.  Recording:
    UHDR_RECORD_REFERENCE=<dir> python -m pytest tests/test_effects_cpu.py tests/test_gpu_effects.py
writes the keys to <dir>/reference_digests.json; copy the "effects/..." entries into that file."""
import json
import os

import uhdr_testlib as T

DIGESTS = os.path.join(T.GOLDEN, "effects_reference_digests.json")
_cache = None


def _recorded(key):
    global _cache
    if _cache is None:
        _cache = json.load(open(DIGESTS)) if os.path.exists(DIGESTS) else {}
    sha = _cache.get(key)
    assert sha is not None, "no recorded reference result for %r in %s" % (key, DIGESTS)
    return sha


def from_reference(key, fn):
    """the reference's answer for `key`: fn() when the reference build is present, else its recorded digest"""
    if T.have_ref():
        v = fn()
        T._record(key, v)
        return v
    return T.Recorded(key, _recorded(key))


def reference_file(key, fn, mine):
    """bytes the reference produced, needed as an input: fn() when the reference build is present (mine() must
    return the same), else mine(), checked against the recorded digest"""
    if T.have_ref():
        v = fn()
        T._record(key, v)
        assert T.same(mine(), v), "%s differs from what the reference produced" % key
        return v
    v = mine()
    assert T.digest(v) == _recorded(key), "%s differs from what the reference produced" % key
    return v
