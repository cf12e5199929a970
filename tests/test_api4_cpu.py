"""Encode API-4 (pre-compressed base image + pre-compressed gain map + metadata -> JPEG/R,
jpegr.cpp:388-434 + appendGainMap :1105-1415) is container work on the host: byte parity with the
reference without a GPU."""
import ctypes as C
import io

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A
from test_probe_cpu import _probe


def _api4(lib, base, gm, md, base_cg=-1, exif=None):
    lib.uhdr_create_encoder.restype = C.c_void_p
    for f in ("uhdr_enc_set_compressed_image", "uhdr_enc_set_gainmap_image", "uhdr_encode", "uhdr_enc_set_exif_data"):
        getattr(lib, f).restype = A.ErrorInfo
    lib.uhdr_get_encoded_stream.restype = C.POINTER(A.CompressedImage)
    enc = C.c_void_p(lib.uhdr_create_encoder())
    try:
        bb, gb = np.frombuffer(base, np.uint8).copy(), np.frombuffer(gm, np.uint8).copy()
        bi = A.CompressedImage(bb.ctypes.data, len(base), len(base), base_cg, -1, -1)
        gi = A.CompressedImage(gb.ctypes.data, len(gm), len(gm), -1, -1, -1)
        e = lib.uhdr_enc_set_compressed_image(enc, C.byref(bi), A.BASE_IMG)
        if e.error_code:
            return ("set_base", e.error_code)
        e = lib.uhdr_enc_set_gainmap_image(enc, C.byref(gi), C.byref(md))
        if e.error_code:
            return ("set_gm", e.error_code)
        if exif is not None:
            xb = np.frombuffer(exif, np.uint8).copy()
            blk = A.MemBlock(xb.ctypes.data, len(exif), len(exif))
            e = lib.uhdr_enc_set_exif_data(enc, C.byref(blk))
            assert e.error_code == 0
        e = lib.uhdr_encode(enc)
        if e.error_code:
            return ("encode", e.error_code)
        o = lib.uhdr_get_encoded_stream(enc).contents
        return C.string_at(o.data, o.data_sz)
    finally:
        lib.uhdr_release_encoder(enc)


@pytest.fixture(scope="module")
def libs(oracle_libs):
    """the product and the reference build (None where it is absent: recorded results stand in)"""
    return C.CDLL(T.GPU_SO), (oracle_libs.Ref().lib if oracle_libs.have_ref() else None)


@pytest.fixture(scope="module")
def parts(libs):
    """base image, gain-map image and metadata of JPEG/R files the reference wrote"""
    mine, ref = libs
    w, h = 192, 128
    hb, sb = T.make_p010(w, h, "smooth"), T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    out = {}
    for name, opts in (("multi", {}), ("single", {"multichannel": 0, "scale": 2})):
        data = T.reference_file("api4/file_192x128_" + name, lambda: T.UhdrApi(ref).encode(hdr, sdr, **opts))
        split = (lambda lib: (lambda p: (p["base_image"], p["gainmap_image"], p["md"]))(_probe(lib, data)))
        out[name] = T.reference_file("api4/parts_192x128_" + name, lambda: split(ref), mine=lambda: split(mine))
    return out


@pytest.mark.parametrize("which", ["multi", "single"])
def test_api4_matches_reference(libs, parts, which):
    mine, ref = libs
    base, gm, md = parts[which]
    a = _api4(mine, base, gm, md)
    assert isinstance(a, bytes), a
    assert T.same(a, T.from_reference("api4/match/" + which, lambda: _api4(ref, base, gm, md)))
    # the result is a JPEG/R both libraries probe identically
    pa = _probe(mine, a)
    pb = T.from_reference("api4/match_probe/" + which, lambda: (lambda p: (p["dims"], p["md"]))(_probe(ref, a)))
    assert T.same((pa["dims"], pa["md"]), pb)


def test_api4_base_without_icc_and_with_exif(libs, parts):
    """a base image from another encoder (Pillow's libjpeg-turbo): no ICC -> one is written from the
    configured gamut; EXIF inside the base image is carried over; unknown gamut is an error"""
    PIL = pytest.importorskip("PIL.Image")
    mine, ref = libs
    _b, gm, md = parts["single"]
    rgb = (np.add.outer(np.arange(128), np.arange(192)) % 256).astype(np.uint8)
    img = PIL.fromarray(np.stack([rgb, rgb[::-1], rgb.T[:128, :192] if False else rgb], -1))
    plain = io.BytesIO()
    img.save(plain, "JPEG", quality=88)
    exif = b"Exif\x00\x00MM\x00\x2a\x00\x00\x00\x08\x00\x00\x00\x00\x00\x00"
    with_exif = io.BytesIO()
    img.save(with_exif, "JPEG", quality=88, exif=exif)
    for bname, base in (("plain", plain.getvalue()), ("exif", with_exif.getvalue())):
        for cg in (A.CG_BT709, A.CG_P3, A.CG_BT2100):
            a = _api4(mine, base, gm, md, cg)
            assert isinstance(a, bytes), a
            assert T.same(a, T.from_reference("api4/pillow_%s/cg%d" % (bname, cg), lambda: _api4(ref, base, gm, md, cg))), cg
        a = _api4(mine, base, gm, md, -1)
        assert not isinstance(a, bytes)   # same error code from both
        assert T.same(a, T.from_reference("api4/pillow_%s/cg-1" % bname, lambda: _api4(ref, base, gm, md, -1)))
    # exif given twice: through the API and inside the base image
    for bname, base in (("exif", with_exif.getvalue()), ("plain", plain.getvalue())):
        a = _api4(mine, base, gm, md, A.CG_BT709, exif=exif)
        assert T.same(a, T.from_reference("api4/pillow_%s/api_exif" % bname, lambda: _api4(ref, base, gm, md, A.CG_BT709, exif=exif)))


def test_api4_rejects_what_the_reference_rejects(libs, parts):
    mine, ref = libs
    base, gm, md = parts["multi"]
    bad = A.GainmapMetadata.from_buffer_copy(bytes(md))
    bad.gamma[1] = -1.0

    def check(name, *args):
        assert T.same(_api4(mine, *args), T.from_reference("api4/reject/" + name, lambda: _api4(ref, *args))), name
    check("bad_gamma", base, gm, bad)
    check("truncated_base", base[:200], gm, md)
    check("not_a_jpeg", b"notajpeg" * 10, gm, md)
    # gain map applied in the alternate image space needs an ICC profile in the gain-map image
    alt = A.GainmapMetadata.from_buffer_copy(bytes(md))
    alt.use_base_cg = 0
    # the gain-map image's APP2 segments: the ISO 21496-1 block, then the ICC profile
    sos = gm.index(b"\xff\xe2")
    while b"ICC_PROFILE" not in gm[sos:sos + 20]:
        sos = gm.index(b"\xff\xe2", sos + 2)
    seglen = (gm[sos + 2] << 8) | gm[sos + 3]
    stripped = gm[:sos] + gm[sos + 2 + seglen:]
    check("alt_space_without_icc", base, stripped, alt)
    check("alt_space", base, gm, alt)
