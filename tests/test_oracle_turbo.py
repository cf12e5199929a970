"""Pins the JPEG side of the checker to the REAL libjpeg-turbo (SURVEY section 8(c) option 2).

oracle/_ref/libuhdr_ref_turbo.so is the reference's own lib/src/jpegencoderhelper.cpp and
jpegdecoderhelper.cpp compiled unmodified against the hand-written libjpeg-62 header
oracle/ref_turbo/jpeglib.h and linked with the libjpeg-turbo binary this image ships (Pillow's).
These tests check that
  * the header's structs have the library's sizes (jpeg_CreateCompress / jpeg_CreateDecompress
    accept them) and streams written through the reference's helper are valid;
  * oracle/jpeg_oracle.c (the restatement used by liboracle.so and by the shim build
    oracle/_ref/libuhdr_ref.so) produces BYTE-IDENTICAL streams to the reference's helper on real
    libjpeg-turbo for every layout the hot path uses -- in particular raw_data_in 4:2:0 with ragged
    sizes (dummy blocks, chroma padding), which Pillow cannot write;
  * whole JPEG/R files and decoded pixels of the two reference builds agree.
Without the reference builds, the C restatement is compared with the digests recorded from the
libjpeg-turbo build (tests/golden/reference_digests.json); the last check needs both builds.
"""
import ctypes as C
import os

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A


def _both_builds():
    return os.path.exists(T.REF_TURBO_SO) and os.path.exists(T.REF_SHIM_SO)


@pytest.fixture(scope="module")
def libs(oracle_libs):
    """(libjpeg-turbo build, shim build, C restatement); the builds are None where oracle/_ref is absent"""
    if oracle_libs.have_ref() and not _both_builds():
        pytest.skip("only one of the two oracle/_ref builds is present")
    if not _both_builds():
        return None, None, oracle_libs.Oracle().lib
    return C.CDLL(T.REF_TURBO_SO), C.CDLL(T.REF_SHIM_SO), oracle_libs.Oracle().lib


def _same_stream(key, mine, turbo, shim, ref_fn):
    """mine (the C restatement's stream) == the libjpeg-turbo build's (live, or its recorded digest); the shim
    build's too where the builds are present"""
    want = T.from_reference("oracle_turbo/" + key, lambda: ref_fn(turbo))
    if not isinstance(want, T.Recorded):
        assert want[:2] == b"\xff\xd8" and want[-2:] == b"\xff\xd9"
        assert ref_fn(shim) == want, ("shim", key)
    assert T.same(mine, want), ("oracle", key)


def _ref_jpeg(lib, img, q, icc=None):
    cap = img.w * img.h * 6 + (1 << 16)
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t()
    iccb = (C.c_uint8 * len(icc)).from_buffer_copy(icc) if icc else None
    rc = lib.ref_jpeg_encode(C.byref(img), q, iccb, C.c_size_t(len(icc) if icc else 0),
                             out.ctypes.data_as(C.c_void_p), C.c_size_t(cap), C.byref(n))
    assert rc == 0
    return bytes(out[:n.value])


SIZES = [(16, 16), (64, 48), (250, 130), (322, 242), (8, 8), (24, 10), (1920, 1080), (1282, 722)]


@pytest.mark.parametrize("w,h", SIZES)
def test_420_raw_data_stream_equals_real_libjpeg_turbo(libs, w, h):
    turbo, shim, olib = libs
    for q, kind in ((95, "noise"), (75, "smooth"), (30, "noise"), (100, "smooth")):
        buf = T.make_yuv420(w, h, kind, seed=w * 7 + h + q)
        img, _k = A.yuv420_image(buf, w, h, A.CG_BT709)
        _same_stream("420/%dx%d/q%d" % (w, h, q), T.oracle_encode(olib, img, q), turbo, shim,
                     lambda lib: _ref_jpeg(lib, img, q))


@pytest.mark.parametrize("w,h", [(64, 48), (250, 130), (333, 77)])
def test_gainmap_streams_equal_real_libjpeg_turbo(libs, w, h):
    turbo, shim, olib = libs
    rs = np.random.RandomState(w + h)
    for q in (95, 60):
        g = rs.randint(0, 256, (h, w)).astype(np.uint8)
        img = A.raw_image(A.FMT_Y400, -1, -1, 1, w, h, [g], [w])
        _same_stream("gainmap_y/%dx%d/q%d" % (w, h, q), T.oracle_encode(olib, img, q, comment=T.GM_COMMENT), turbo, shim,
                     lambda lib: _ref_jpeg(lib, img, q))
        rgb = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        img = A.raw_image(A.FMT_RGB888, -1, -1, 1, w, h, [rgb], [w])
        _same_stream("gainmap_rgb/%dx%d/q%d" % (w, h, q), T.oracle_encode(olib, img, q, comment=T.GM_COMMENT), turbo, shim,
                     lambda lib: _ref_jpeg(lib, img, q))


@pytest.mark.parametrize("w,h,kind", [(256, 128, "smooth"), (250, 130, "noise"), (1280, 720, "noise")])
def test_whole_files_and_decodes_agree(libs, w, h, kind):
    turbo, shim, _o = libs
    if turbo is None:
        pytest.skip("compares the two reference builds with each other: needs oracle/_ref")
    ta, sa = T.UhdrApi(turbo), T.UhdrApi(shim)
    hb, sb = T.make_p010(w, h, kind), T.make_yuv420(w, h, kind)
    hdr, _k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, _k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    for api1 in (True, False):
        a = ta.encode(hdr, sdr if api1 else None)
        assert a == sa.encode(hdr, sdr if api1 else None)
        pa, pb = ta.decode(a), sa.decode(a)
        assert (pa[0] == pb[0]).all() and (pa[1] == pb[1]).all() and T.md_equal(pa[2], pb[2])
        pa, pb = ta.decode(a, A.FMT_RGBA1010102, A.CT_PQ), sa.decode(a, A.FMT_RGBA1010102, A.CT_PQ)
        assert (pa[0] == pb[0]).all()
        pa, pb = ta.decode(a, A.FMT_RGBA8888, A.CT_SRGB), sa.decode(a, A.FMT_RGBA8888, A.CT_SRGB)
        assert (pa[0] == pb[0]).all()
