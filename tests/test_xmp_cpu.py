"""Gain-map metadata in hdrgm XMP form (Ultra HDR v1 files, Apple's variant): the host-side reader of
libuhdr_b200 against the reference's getMetadataFromXMP (jpegrutils.cpp:646-874) through
uhdr_dec_probe.  No GPU needed: probing is host work."""
import ctypes as C
import os

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A
from test_probe_cpu import _probe

APPLE = ["apple_gainmap_new.jpg", "apple_gainmap_old.jpg"]   # the reference's own fixtures (tests/data), in tests/golden/
FIELDS = ("max_content_boost", "min_content_boost", "gamma", "offset_sdr", "offset_hdr", "hdr_capacity_min", "hdr_capacity_max")


def _vals(md, with_cg=True):
    out = []
    for f in FIELDS:
        v = getattr(md, f)
        out.append(tuple(np.float32(x).tobytes() for x in v) if hasattr(v, "__len__") else np.float32(v).tobytes())
    if with_cg:
        out.append(int(md.use_base_cg) != 0)
    return out


@pytest.fixture(scope="module")
def libs(oracle_libs):
    """the product and the reference build (None where it is absent: recorded results stand in)"""
    return C.CDLL(T.GPU_SO), (oracle_libs.Ref().lib if oracle_libs.have_ref() else None)


def _probe_summary(p, with_cg=True):
    if "error" in p:
        return ("error", p["error"])
    return (p["dims"], p["exif"], p["icc"], p["base_image"], p["gainmap_image"], _vals(p["md"], with_cg))


@pytest.mark.parametrize("path", APPLE)
def test_apple_fixtures(libs, path):
    """the reference's own Apple fixtures (tests/jpegr_test.cpp:1518-1562): XMP element HDRGainMapHeadroom
    or, failing that, the headroom derived from the EXIF maker notes"""
    mine, ref = libs
    data = open(os.path.join(T.GOLDEN, path), "rb").read()
    a = _probe(mine, data)
    assert "error" not in a, a.get("error")
    # use_base_cg: the reference never initialises it on the Apple branch
    b = T.from_reference("xmp/apple/" + path, lambda: _probe_summary(_probe(ref, data), False))
    assert T.same(_probe_summary(a, False), b)
    lib = mine
    lib.is_uhdr_image.argtypes = [C.c_void_p, C.c_int]
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    assert lib.is_uhdr_image(buf, len(data)) == 1


def _xmp_only_file(ref_lib, attrs, extra=""):
    """a JPEG/R written by the reference whose gain-map image carries an hdrgm XMP packet instead of the
    ISO 21496-1 block"""
    w, h = 128, 64
    hb, sb = T.make_p010(w, h, "smooth"), T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    data = T.reference_file("xmp/file_128x64", lambda: T.UhdrApi(ref_lib).encode(hdr, sdr))
    sig = b"urn:iso:std:iso:ts:21496:-1\x00"
    second = data.index(b"\xff\xd8", 4 + data.index(b"\xff\xd9") - 2) if False else None
    # the gain-map image is the last SOI that is followed by APP2/ISO with a payload
    gpos = data.rindex(b"\xff\xd8\xff")
    g = data[gpos:]
    i = g.index(b"\xff\xe2", 2)
    while sig not in g[i:i + 40]:
        i = g.index(b"\xff\xe2", i + 2)
    seglen = (g[i + 2] << 8) | g[i + 3]
    body = '<x:xmpmeta xmlns:x="adobe:ns:meta/" x:xmptk="Adobe XMP Core 5.1.2"><rdf:RDF ' \
           'xmlns:rdf="http://www.w3.org/1999/02/22-rdf-syntax-ns#"><rdf:Description ' \
           'xmlns:hdrgm="http://ns.adobe.com/hdr-gain-map/1.0/" ' + \
           " ".join('%s="%s"' % kv for kv in attrs) + ">" + extra + "</rdf:Description></rdf:RDF></x:xmpmeta>"
    payload = b"http://ns.adobe.com/xap/1.0/\x00" + body.encode()
    app1 = b"\xff\xe1" + (len(payload) + 2).to_bytes(2, "big") + payload
    g2 = g[:i] + app1 + g[i + 2 + seglen:]
    return data[:gpos] + g2


FULL = [("hdrgm:Version", "1.0"), ("hdrgm:GainMapMin", "-0.25"), ("hdrgm:GainMapMax", "2.5"), ("hdrgm:Gamma", "1.25"),
        ("hdrgm:OffsetSDR", "0.015625"), ("hdrgm:OffsetHDR", "0.03125"), ("hdrgm:HDRCapacityMin", "0"),
        ("hdrgm:HDRCapacityMax", "2.3"), ("hdrgm:BaseRenditionIsHDR", "False")]


@pytest.mark.parametrize("case", ["full", "required_only", "no_version", "no_max", "no_capmax", "bad_gamma", "hdr_base",
                                  "bad_bool", "capmax_below_min", "neg_offset"])
def test_hdrgm_xmp_metadata(libs, case):
    mine, ref = libs
    attrs = list(FULL)
    drop = {"required_only": ("GainMapMin", "Gamma", "OffsetSDR", "OffsetHDR", "HDRCapacityMin", "BaseRenditionIsHDR"),
            "no_version": ("Version",), "no_max": ("GainMapMax",), "no_capmax": ("HDRCapacityMax",)}.get(case, ())
    attrs = [(k, v) for k, v in attrs if k.split(":")[1] not in drop]
    sub = {"bad_gamma": ("hdrgm:Gamma", "abc"), "hdr_base": ("hdrgm:BaseRenditionIsHDR", "True"),
           "bad_bool": ("hdrgm:BaseRenditionIsHDR", "maybe"), "capmax_below_min": ("hdrgm:HDRCapacityMax", "-1"),
           "neg_offset": ("hdrgm:OffsetSDR", "-0.5")}.get(case)
    if sub:
        attrs = [(k, sub[1] if k == sub[0] else v) for k, v in attrs]
    data = _xmp_only_file(ref, attrs)
    a = _probe(mine, data)
    summary = (lambda p: ("error", p["error"]) if "error" in p else _vals(p["md"]))
    b = T.from_reference("xmp/hdrgm/" + case, lambda: summary(_probe(ref, data)))
    assert T.same(summary(a), b), (case, a.get("error"), b)
