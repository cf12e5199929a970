"""Image effects of the C API (uhdr_add_effect_*) on the device, against the reference's C API: whole encoded
files byte for byte, decoded pixels / gain maps / metadata / descriptors, and the error codes of the encoder's
and decoder's validation of sizes."""
import ctypes as C

import numpy as np
import pytest

import effects_testlib as E
import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A

pytestmark = pytest.mark.gpu

INVALID_PARAM, INVALID_OPERATION = 3, 5


@pytest.fixture(scope="module")
def ref(oracle_libs):
    """the reference build's library, or None where recorded results stand in"""
    return oracle_libs.Ref().lib if oracle_libs.have_ref() else None


def _decl(lib):
    T.UhdrApi(lib)
    for f in ("uhdr_add_effect_mirror", "uhdr_add_effect_rotate", "uhdr_add_effect_crop", "uhdr_add_effect_resize",
              "uhdr_enc_set_compressed_image"):
        getattr(lib, f).restype = A.ErrorInfo
    lib.uhdr_add_effect_crop.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]


def _add(lib, h, effects):
    """-> 0, or the first failing call's error code"""
    for e in effects:
        fn = getattr(lib, "uhdr_add_effect_" + e[0])
        code = fn(h, *e[1:]).error_code
        if code:
            return code
    return 0


# ------------------------------------------------------------------------------------------------
# encoder
# ------------------------------------------------------------------------------------------------
def _inputs(cfg):
    """name -> (w, h, hdr image, sdr image or None, encode options); buffers kept alive in the tuple"""
    kind, w, h = cfg
    if kind in ("p010", "p010_420"):
        hb = T.make_p010(w, h, "smooth")
        hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
        sdr = k2 = None
        if kind == "p010_420":
            sb = T.make_yuv420(w, h, "smooth")
            sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
        return hdr, sdr, (hb, k1, k2)
    if kind == "f16_8888":
        hb, sb = T.make_rgbaf16(w, h), T.make_rgba8888(w, h)
        hdr = A.raw_image(A.FMT_RGBAF16, A.CG_BT2100, A.CT_LINEAR, A.CR_FULL, w, h, [hb], [w])
        sdr = A.raw_image(A.FMT_RGBA8888, A.CG_BT709, A.CT_SRGB, A.CR_FULL, w, h, [sb], [w])
        return hdr, sdr, (hb, sb)
    if kind == "1010102":  # smooth: noise this small does not fit the reference's output buffer (w*h*6 bytes)
        yy, xx = np.mgrid[0:h, 0:w]
        r = 512 + 400 * np.sin(xx / 37.0)
        g = 512 + 400 * np.cos(yy / 23.0)
        b = (xx + yy) * 1023.0 / (w + h)
        hb = (r.astype(np.uint32) | g.astype(np.uint32) << 10 | b.astype(np.uint32) << 20 | np.uint32(3 << 30)).ravel()
        hdr = A.raw_image(A.FMT_RGBA1010102, A.CG_BT2100, A.CT_PQ, A.CR_FULL, w, h, [hb], [w])
        return hdr, None, (hb,)
    raise ValueError(kind)


def _encode(lib, cfg, effects, scale=1, multichannel=1, rearm=False):
    """the encoded file, or (stage, error code)"""
    _decl(lib)
    hdr, sdr, keep = _inputs(cfg)
    L = lib
    enc = C.c_void_p(L.uhdr_create_encoder())
    try:
        assert L.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG).error_code == 0
        if sdr is not None:
            assert L.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG).error_code == 0
        assert L.uhdr_enc_set_gainmap_scale_factor(enc, scale).error_code == 0
        assert L.uhdr_enc_set_using_multi_channel_gainmap(enc, multichannel).error_code == 0
        code = _add(L, enc, effects)
        if code:
            return ("add", code)
        e = L.uhdr_encode(enc)
        if e.error_code:
            return ("encode", e.error_code)
        o = L.uhdr_get_encoded_stream(enc).contents
        out = C.string_at(o.data, o.data_sz)
        if rearm:  # the resident inputs were not touched by the effects: the same bytes again
            assert L.uhdr_b200_enc_rearm(enc) == 0
            assert L.uhdr_encode(enc).error_code == 0
            o = L.uhdr_get_encoded_stream(enc).contents
            assert C.string_at(o.data, o.data_sz) == out
        return out
    finally:
        L.uhdr_release_encoder(enc)
        del keep


def _singles(w, h):
    return {
        "mirror_h": [("mirror", 1)],
        "mirror_v": [("mirror", 0)],
        "rotate_90": [("rotate", 90)],
        "rotate_180": [("rotate", 180)],
        "rotate_270": [("rotate", 270)],
        "crop_odd_origin": [("crop", 3, 3 + ((w - 10) & ~1), 5, 5 + ((h - 12) & ~1))],
        "downscale": [("resize", (w // 3) & ~1, (h // 3) & ~1)],
        "upscale": [("resize", 2 * w, 2 * h)],
        # rotate 90 -> crop -> mirror -> resize
        "chain": [("rotate", 90), ("crop", 1, 1 + ((h - 6) & ~1), 3, 3 + ((w - 8) & ~1)), ("mirror", 1),
                  ("resize", ((h - 6) // 2) & ~1, ((w - 8) // 2) & ~1)],
    }


ENC_CASES = []
for _cfg, _opts in ((("p010", 256, 128), {}), (("p010_420", 256, 128), {}), (("p010", 650, 370), {}),
                    (("p010_420", 650, 370), {}), (("f16_8888", 256, 128), {}), (("1010102", 256, 128), {}),
                    (("p010_420", 650, 370), {"scale": 4, "multichannel": 0})):
    for _name, _fx in _singles(_cfg[1], _cfg[2]).items():
        ENC_CASES.append(pytest.param(_cfg, _opts, _fx, id="%s_%dx%d%s-%s" % (_cfg + ("_s4" if _opts else "", _name))))
# chains that end below the 8x8 minimum of uhdr_enc_set_raw_image: not checked again, the reference encodes them
for _cfg in (("p010", 256, 128), ("p010_420", 256, 128)):
    ENC_CASES.append(pytest.param(_cfg, {}, [("rotate", 90), ("resize", 2, 2)], id="%s_%dx%d-to_2x2" % _cfg))
    ENC_CASES.append(pytest.param(_cfg, {}, [("crop", 10, 14, 6, 10), ("mirror", 0)], id="%s_%dx%d-to_4x4" % _cfg))
ENC_CASES.append(pytest.param(("p010_420", 3840, 2160), {}, [("rotate", 90), ("crop", 100, 2100, 300, 3500)],
                              id="p010_420_3840x2160-rotate_crop"))


def _key(parts):
    return "effects/" + "/".join(str(p) for p in parts)


@pytest.mark.parametrize("cfg,opts,effects", ENC_CASES)
def test_encode_with_effects_matches_reference(gpu, ref, cfg, opts, effects):
    mine = _encode(gpu.lib, cfg, effects, rearm=True, **opts)
    assert isinstance(mine, bytes), mine
    want = E.from_reference(_key(("enc",) + cfg + tuple(sorted(opts.items())) + (repr(effects),)),
                            lambda: _encode(ref, cfg, effects, **opts))
    assert T.same(mine, want)


ENC_ERRORS = {
    "crop_empty_width": (("p010_420", 256, 128), [("crop", 300, 400, 0, 64)]),
    "crop_empty_height": (("p010_420", 256, 128), [("crop", 0, 64, 64, 64)]),
    "crop_odd_width_p010": (("p010", 256, 128), [("crop", 0, 63, 0, 64)]),
    "crop_odd_height_p010": (("p010", 256, 128), [("crop", 0, 64, 1, 64)]),
    "crop_odd_width_rgba": (("f16_8888", 256, 128), [("crop", 0, 63, 0, 63)]),   # allowed: packed formats only
    "crop_clamped": (("1010102", 256, 128), [("crop", -7, 1000, -3, 1000)]),
    "resize_zero": (("p010_420", 256, 128), [("resize", 0, 64)]),
    "resize_too_large": (("p010_420", 256, 128), [("resize", 8194, 64)]),
    "resize_odd_p010": (("p010", 256, 128), [("resize", 63, 64)]),
    "resize_odd_rgba": (("1010102", 256, 128), [("resize", 63, 65)]),           # allowed
    "crop_after_rotate": (("p010_420", 256, 128), [("rotate", 270), ("crop", 0, 200, 0, 200)]),  # clamps to 128 x 200
}


@pytest.mark.parametrize("name", sorted(ENC_ERRORS))
def test_encoder_size_checks_match_reference(gpu, ref, name):
    cfg, effects = ENC_ERRORS[name]
    mine = _encode(gpu.lib, cfg, effects)
    want = E.from_reference(_key(("enc_check", name)), lambda: _encode(ref, cfg, effects))
    assert T.same(mine, want)
    if name.startswith(("crop_empty", "crop_odd_width_p", "crop_odd_height", "resize_zero", "resize_too", "resize_odd_p")):
        assert mine == ("encode", INVALID_PARAM)
    else:
        assert isinstance(mine, bytes)


def _compressed_sdr_encode(lib, with_raw_sdr):
    """API-2 / API-3 with an effect: refused before any pixel work"""
    _decl(lib)
    w, h = 256, 128
    hdr, sdr, keep = _inputs(("p010_420", w, h))
    jpg = T.oracle_encode(C.CDLL(T.ORACLE_SO), sdr, 90)  # any baseline JPEG of the SDR intent
    jb = np.frombuffer(jpg, np.uint8).copy()
    enc = C.c_void_p(lib.uhdr_create_encoder())
    try:
        assert lib.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG).error_code == 0
        if with_raw_sdr:
            assert lib.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG).error_code == 0
        ci = A.CompressedImage(jb.ctypes.data, len(jpg), len(jpg), A.CG_BT709, -1, -1)
        assert lib.uhdr_enc_set_compressed_image(enc, C.byref(ci), A.SDR_IMG).error_code == 0
        assert _add(lib, enc, [("mirror", 1)]) == 0
        first = lib.uhdr_encode(enc).error_code
        lib.uhdr_reset_encoder(enc)   # the list goes with the reset
        assert lib.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG).error_code == 0
        if with_raw_sdr:
            assert lib.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG).error_code == 0
        assert lib.uhdr_enc_set_compressed_image(enc, C.byref(ci), A.SDR_IMG).error_code == 0
        return first, lib.uhdr_encode(enc).error_code
    finally:
        lib.uhdr_release_encoder(enc)
        del keep


@pytest.mark.parametrize("with_raw_sdr", [False, True], ids=["api3", "api2"])
def test_effects_with_compressed_sdr_are_refused(gpu, ref, with_raw_sdr):
    mine = _compressed_sdr_encode(gpu.lib, with_raw_sdr)
    assert mine == (INVALID_OPERATION, 0)
    want = E.from_reference(_key(("enc_compressed", with_raw_sdr)), lambda: _compressed_sdr_encode(ref, with_raw_sdr))
    assert T.same(mine, want)


# ------------------------------------------------------------------------------------------------
# decoder
# ------------------------------------------------------------------------------------------------
DEC_FILES = {  # name -> (encoder input, options): 650x370 with a scale-4 map (ratio 650/162 = 4.0123), 640x368 default
    "650x370_s4": (("p010_420", 650, 370), {"scale": 4, "multichannel": 0}),
    "640x368": (("p010_420", 640, 368), {}),
    "3840x2160": (("p010_420", 3840, 2160), {}),
}
OUTPUTS = {"f16_linear": (A.FMT_RGBAF16, A.CT_LINEAR), "1010102_pq": (A.FMT_RGBA1010102, A.CT_PQ),
           "1010102_hlg": (A.FMT_RGBA1010102, A.CT_HLG), "8888_srgb": (A.FMT_RGBA8888, A.CT_SRGB)}


@pytest.fixture(scope="module")
def files(gpu, ref):
    cache = {}

    def get(name):
        if name not in cache:
            cfg, opts = DEC_FILES[name]
            cache[name] = E.reference_file(_key(("dec_file", name)), lambda: _encode(ref, cfg, [], **opts),
                                           mine=lambda: _encode(gpu.lib, cfg, [], **opts))
        return cache[name]
    return get


def _decode(lib, data, effects, out, probe_first=False):
    """(pixels, gain map, metadata, image descriptor, map descriptor), or (stage, error code)"""
    _decl(lib)
    L = lib
    fmt, ct = OUTPUTS[out]
    dec = C.c_void_p(L.uhdr_create_decoder())
    try:
        buf = np.frombuffer(data, np.uint8).copy()
        ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
        assert L.uhdr_dec_set_image(dec, C.byref(ci)).error_code == 0
        assert L.uhdr_dec_set_out_img_format(dec, fmt).error_code == 0
        assert L.uhdr_dec_set_out_color_transfer(dec, ct).error_code == 0
        if probe_first:  # effects may still be added after a probe: the handle has not sailed
            assert L.uhdr_dec_probe(dec).error_code == 0
        code = _add(L, dec, effects)
        if code:
            return ("add", code)
        e = L.uhdr_decode(dec)
        if e.error_code:
            return ("decode", e.error_code)
        assert _add(L, dec, [("rotate", 90)]) == INVALID_OPERATION
        d = L.uhdr_get_decoded_image(dec).contents
        bpp = 8 if fmt == A.FMT_RGBAF16 else 4
        px = np.ctypeslib.as_array(C.cast(d.planes[0], C.POINTER(C.c_uint8)), (d.h, d.stride[0] * bpp))[:, :d.w * bpp].copy()
        g = L.uhdr_get_decoded_gainmap_image(dec).contents
        gb = 1 if g.fmt == A.FMT_Y400 else 4
        gm = np.ctypeslib.as_array(C.cast(g.planes[0], C.POINTER(C.c_uint8)), (g.h, g.stride[0] * gb))[:, :g.w * gb].copy()
        md = bytes(L.uhdr_dec_get_gainmap_metadata(dec).contents)
        return px, gm, md, (d.w, d.h, d.stride[0], d.fmt, d.cg), (g.w, g.h, g.stride[0], g.fmt)
    finally:
        L.uhdr_release_decoder(dec)


DEC_CASES = []
for _file, (_cfg, _o) in DEC_FILES.items():
    if _file == "3840x2160":
        continue
    for _name, _fx in _singles(_cfg[1], _cfg[2]).items():
        for _out in OUTPUTS:
            DEC_CASES.append(pytest.param(_file, _out, _fx, id="%s-%s-%s" % (_file, _name, _out)))
DEC_CASES.append(pytest.param("3840x2160", "f16_linear", [("rotate", 90)], id="3840x2160-rotate_90-f16_linear"))


@pytest.mark.parametrize("file,out,effects", DEC_CASES)
def test_decode_with_effects_matches_reference(gpu, ref, files, file, out, effects):
    data = files(file)
    mine = _decode(gpu.lib, data, effects, out)
    assert isinstance(mine, tuple) and len(mine) == 5, mine
    px, gm, md, d, g = mine
    assert d[2] == (d[0] + 63) // 64 * 64 and g[2] == (g[0] + 63) // 64 * 64  # stride ALIGNM(w, 64) after effects
    want = E.from_reference(_key(("dec", file, out, repr(effects))), lambda: _decode(ref, data, effects, out))
    assert T.same(mine, want)


def test_decode_effects_added_after_probe(gpu, ref, files):
    data = files("650x370_s4")
    effects = _singles(650, 370)["chain"]
    mine = _decode(gpu.lib, data, effects, "f16_linear", probe_first=True)
    assert isinstance(mine, tuple) and len(mine) == 5, mine
    assert T.same(mine, E.from_reference(_key(("dec", "650x370_s4", "f16_linear", repr(effects))),
                                         lambda: _decode(ref, data, effects, "f16_linear")))


def test_decode_without_effects_keeps_the_plain_descriptors(gpu, files):
    px, gm, md, d, g = _decode(gpu.lib, files("650x370_s4"), [], "f16_linear")
    assert d == (650, 370, 650, A.FMT_RGBAF16, d[4]) and g[:3] == (162, 92, 162)


DEC_ERRORS = {
    "crop_empty_on_map": [("crop", 1, 3, 0, 370)],      # (int)(3 / 4.0123) == 0 columns of the map
    "resize_empty_on_map": [("resize", 3, 3)],
    "crop_empty": [("crop", 700, 800, 0, 10)],
    "resize_too_large": [("resize", 8200, 100)],
}


@pytest.mark.parametrize("name", sorted(DEC_ERRORS))
def test_decoder_size_checks_match_reference(gpu, ref, files, name):
    data = files("650x370_s4")
    effects = DEC_ERRORS[name]
    mine = _decode(gpu.lib, data, effects, "f16_linear")
    assert mine == ("decode", INVALID_PARAM)
    assert T.same(mine, E.from_reference(_key(("dec_check", name)), lambda: _decode(ref, data, effects, "f16_linear")))
