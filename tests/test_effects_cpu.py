"""Image effects of the C API (uhdr_add_effect_*) where no device is needed: argument checks, the sailed state
after a host-only API-4 encode, and effects refused with compressed intents.  Error codes equal the reference's."""
import ctypes as C

import numpy as np
import pytest

import effects_testlib as E
import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A
from test_api4_cpu import _api4, libs, parts  # noqa: F401  (fixtures)

INVALID_PARAM, INVALID_OPERATION = 3, 5


def _decl(lib):
    lib.uhdr_create_encoder.restype = C.c_void_p
    lib.uhdr_create_decoder.restype = C.c_void_p
    for f in ("uhdr_add_effect_mirror", "uhdr_add_effect_rotate", "uhdr_add_effect_crop", "uhdr_add_effect_resize",
              "uhdr_enc_set_compressed_image", "uhdr_enc_set_gainmap_image", "uhdr_encode"):
        getattr(lib, f).restype = A.ErrorInfo
    lib.uhdr_add_effect_mirror.argtypes = [C.c_void_p, C.c_int]
    lib.uhdr_add_effect_rotate.argtypes = [C.c_void_p, C.c_int]
    lib.uhdr_add_effect_crop.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.uhdr_add_effect_resize.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.uhdr_get_encoded_stream.restype = C.POINTER(A.CompressedImage)


def _add_all(lib, h):
    """one call of each kind with valid arguments -> their error codes"""
    return (lib.uhdr_add_effect_mirror(h, 0).error_code, lib.uhdr_add_effect_rotate(h, 90).error_code,
            lib.uhdr_add_effect_crop(h, 0, 8, 0, 8).error_code, lib.uhdr_add_effect_resize(h, 16, 16).error_code)


def _argument_codes(lib):
    _decl(lib)
    codes = [_add_all(lib, None)]
    for create, release in ((lib.uhdr_create_encoder, lib.uhdr_release_encoder),
                            (lib.uhdr_create_decoder, lib.uhdr_release_decoder)):
        h = C.c_void_p(create())
        try:
            codes.append(tuple(lib.uhdr_add_effect_mirror(h, d).error_code for d in (-1, 0, 1, 2)))
            codes.append(tuple(lib.uhdr_add_effect_rotate(h, d).error_code for d in (0, 45, 90, 180, 270, 360, -90)))
            # sizes are not looked at before the handle sails
            codes.append((lib.uhdr_add_effect_crop(h, -5, -9, 100, 2).error_code,
                          lib.uhdr_add_effect_resize(h, 0, -1).error_code,
                          lib.uhdr_add_effect_resize(h, 100000, 3).error_code))
        finally:
            release(h)
    return tuple(codes)


def test_add_effect_argument_errors(libs):
    mine, ref = libs
    got = _argument_codes(mine)
    assert got[0] == (INVALID_PARAM,) * 4
    assert got[1] == (INVALID_PARAM, 0, 0, INVALID_PARAM)
    assert got[2] == (INVALID_PARAM, INVALID_PARAM, 0, 0, 0, INVALID_PARAM, INVALID_PARAM)
    assert T.same(got, E.from_reference("effects/cpu/argument_codes", lambda: _argument_codes(ref)))


def _api4_with_effects(lib, base, gm, md, add_before_encode):
    """(set, encode, add-after-sail codes, and after reset: a plain API-4 encode of the same parts)"""
    _decl(lib)
    enc = C.c_void_p(lib.uhdr_create_encoder())
    try:
        def configure():
            bb, gb = np.frombuffer(base, np.uint8).copy(), np.frombuffer(gm, np.uint8).copy()
            bi = A.CompressedImage(bb.ctypes.data, len(base), len(base), -1, -1, -1)
            gi = A.CompressedImage(gb.ctypes.data, len(gm), len(gm), -1, -1, -1)
            assert lib.uhdr_enc_set_compressed_image(enc, C.byref(bi), A.BASE_IMG).error_code == 0
            assert lib.uhdr_enc_set_gainmap_image(enc, C.byref(gi), C.byref(md)).error_code == 0
            return bb, gb
        keep = configure()
        added = _add_all(lib, enc) if add_before_encode else ()
        first = lib.uhdr_encode(enc).error_code
        after = _add_all(lib, enc)
        again = lib.uhdr_encode(enc).error_code  # the cached status
        lib.uhdr_reset_encoder(enc)
        keep = configure()
        e = lib.uhdr_encode(enc)
        out = C.string_at(lib.uhdr_get_encoded_stream(enc).contents.data,
                          lib.uhdr_get_encoded_stream(enc).contents.data_sz) if e.error_code == 0 else e.error_code
        del keep
        return added, first, after, again, out
    finally:
        lib.uhdr_release_encoder(enc)


@pytest.mark.parametrize("add_before_encode", [False, True])
def test_api4_sailed_and_compressed_intent(libs, parts, add_before_encode):
    mine, ref = libs
    base, gm, md = parts["multi"]
    got = _api4_with_effects(mine, base, gm, md, add_before_encode)
    added, first, after, again, out = got
    if add_before_encode:
        # effects with a compressed intent: refused when the handle sails
        assert added == (0, 0, 0, 0) and first == INVALID_OPERATION and again == INVALID_OPERATION
    else:
        assert first == 0 and again == 0
    assert after == (INVALID_OPERATION,) * 4
    # reset clears the list: the same API-4 encode then succeeds and writes what it writes without effects
    assert isinstance(out, bytes) and out == _api4(mine, base, gm, md)
    assert T.same(got, E.from_reference("effects/cpu/api4_sailed/%d" % add_before_encode,
                                        lambda: _api4_with_effects(ref, base, gm, md, add_before_encode)))
