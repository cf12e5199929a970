"""Device entropy decoder (huffdec.cu) vs the host decoder and the CPU checker: decoded planes must
be identical for every sampling layout, size (whole and ragged MCUs, dummy edge blocks), quality and
content, and the device path must really have run (no silent hand-back to the host decoder)."""
import ctypes as C

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A
from test_gpu_jpeg_api import _img

pytestmark = pytest.mark.gpu

CASES = [  # fmt, w, h, kind, quality
    (A.FMT_YUV420, 64, 48, "noise", 95), (A.FMT_YUV420, 320, 240, "smooth", 90), (A.FMT_YUV420, 1280, 720, "noise", 95),
    (A.FMT_YUV420, 1280, 720, "smooth", 30), (A.FMT_YUV420, 72, 34, "noise", 100), (A.FMT_YUV420, 1000, 562, "smooth", 75),
    (A.FMT_Y400, 64, 48, "noise", 95), (A.FMT_Y400, 72, 33, "smooth", 50), (A.FMT_Y400, 960, 540, "noise", 85),
    (A.FMT_RGB888, 64, 48, "noise", 95), (A.FMT_RGB888, 100, 61, "smooth", 95), (A.FMT_RGB888, 960, 540, "noise", 95),
    (A.FMT_RGB888, 960, 540, "smooth", 12), (A.FMT_YUV444, 96, 40, "noise", 95),
]


def _stats(lib):
    st = (C.c_ulonglong * 3)()
    lib.uhdr_b200_entropy_decoder_stats(st)
    return list(st)


def _decode(lib, data, mode, w, h):
    buf = np.zeros(w * h * 4 + 65536, np.uint8)
    out = A.raw_image(-1, -1, -1, -1, 0, 0, [buf], [0])
    cbuf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    rc = lib.uhdr_b200_jpeg_decode(cbuf, C.c_size_t(len(data)), mode, C.byref(out), C.c_size_t(buf.size))
    return rc, out, buf


@pytest.mark.parametrize("case", CASES, ids=lambda c: "fmt%d_%dx%d_%s_q%d" % c)
def test_device_entropy_decoder_matches_host(gpu, oracle_libs, case):
    fmt, w, h, kind, q = case
    o = oracle_libs.Oracle().lib
    lib = gpu.lib
    lib.uhdr_b200_entropy_decoder_stats.restype = None
    img, keep = _img(fmt, w, h, kind)
    data = T.oracle_encode(o, img, q)
    mode = 0 if fmt in (A.FMT_YUV420, A.FMT_YUV444) else 2
    prev = lib.uhdr_b200_set_entropy_decoder(1)
    try:
        rc, out_h, buf_h = _decode(lib, data, mode, w, h)
        assert rc == 0, T.gpu_err(gpu)
        s0 = _stats(lib)
        lib.uhdr_b200_set_entropy_decoder(2)
        rc, out_d, buf_d = _decode(lib, data, mode, w, h)
        assert rc == 0, T.gpu_err(gpu)
        s1 = _stats(lib)
    finally:
        lib.uhdr_b200_set_entropy_decoder(prev)
    assert s1[0] == s0[0] + 1 and s1[1] == s0[1], ("device decoder did not run", s0, s1)
    assert out_d.fmt == out_h.fmt and out_d.w == out_h.w and out_d.h == out_h.h
    assert (buf_d == buf_h).all(), (case, int((buf_d != buf_h).sum()), s1)
    # and against the CPU checker (luma plane is enough here; test_decode_planes covers the layout)
    hd, planes = T.oracle_decode(o, data)
    if mode == 0 or hd.frame.ncomp == 1:
        assert (buf_d[:w * h].reshape(h, w) == planes[0][:h, :w]).all()


def test_device_entropy_decoder_whole_file(gpu, oracle_libs):
    """uhdr_decode of a JPEG/R with both entropy decoders -> identical pixels"""
    api = T.UhdrApi(gpu.lib)
    w, h = 1280, 720
    hb = T.make_p010(w, h, "smooth")
    sb = T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    data = api.encode(hdr, sdr)
    lib = gpu.lib
    lib.uhdr_b200_entropy_decoder_stats.restype = None
    prev = lib.uhdr_b200_set_entropy_decoder(1)
    try:
        a = api.decode(data)
        s0 = _stats(lib)
        lib.uhdr_b200_set_entropy_decoder(2)
        b = api.decode(data)
        s1 = _stats(lib)
    finally:
        lib.uhdr_b200_set_entropy_decoder(prev)
    assert s1[0] == s0[0] + 2 and s1[1] == s0[1], (s0, s1)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_device_entropy_decoder_4k_against_reference(gpu, oracle_libs):
    """config 4 geometry: a 3840x2160 file (≈50k subsequences per scan, both scans decoded concurrently on
    two streams) -> pixels, gain map and metadata identical to the reference decoder's."""
    import bench
    w, h = 3840, 2160
    p, y = bench.make_frame(w, h, 3)
    hdr, sdr, keep = bench.frame_descs(p, y, w, h)
    mine = T.UhdrApi(gpu.lib)
    ref = T.UhdrApi(oracle_libs.Ref().lib) if oracle_libs.have_ref() else None
    data = mine.encode(hdr, sdr)
    lib = gpu.lib
    lib.uhdr_b200_entropy_decoder_stats.restype = None
    s0 = _stats(lib)
    pa, ga, ma, cga = mine.decode(data)
    s1 = _stats(lib)
    assert s1[0] == s0[0] + 2 and s1[1] == s0[1], (s0, s1)
    # recorded results describe the reference's decode of the reference's own file: the stream must be that file
    assert T.same(data, T.from_reference("huffdec/4k_file", lambda: ref.encode(hdr, sdr)))
    assert T.same((pa, ga, ma, cga), T.from_reference("huffdec/4k_decoded", lambda: ref.decode(data)))


def test_corrupted_scans_agree_with_host_decoder(gpu, oracle_libs):
    """bytes flipped inside the entropy-coded segments: whatever the host decoder makes of the stream
    (an error, or garbage pixels), the device decoder must make the same of it -- and never hang."""
    api = T.UhdrApi(gpu.lib)
    lib = gpu.lib
    w, h = 640, 368
    hb = T.make_p010(w, h, "smooth")
    sb = T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    good = bytearray(api.encode(hdr, sdr))
    sos = [i for i in range(len(good) - 1) if good[i] == 0xFF and good[i + 1] == 0xDA]
    assert len(sos) == 2
    rs = np.random.RandomState(99)

    def run(data, mode):
        prev = lib.uhdr_b200_set_entropy_decoder(mode)
        try:
            dec = C.c_void_p(lib.uhdr_create_decoder())
            buf = np.frombuffer(bytes(data), np.uint8).copy()
            ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
            e = lib.uhdr_dec_set_image(dec, C.byref(ci))
            if e.error_code == 0:
                e = lib.uhdr_decode(dec)
            px = None
            if e.error_code == 0:
                d = lib.uhdr_get_decoded_image(dec).contents
                px = np.ctypeslib.as_array(C.cast(d.planes[0], C.POINTER(C.c_uint8)), (d.h, d.stride[0] * 8)).copy()
            lib.uhdr_release_decoder(dec)
            return e.error_code, px
        finally:
            lib.uhdr_b200_set_entropy_decoder(prev)

    for t in range(24):
        bad = bytearray(good)
        s = sos[t % 2]
        lo = s + 16
        hi = (sos[1] - 64) if t % 2 == 0 else (len(bad) - 8)
        for _ in range(1 + t % 3):
            pos = int(rs.randint(lo, hi))
            v = int(rs.randint(0, 255))
            bad[pos] = v if v != 0xFF else 0x7F   # keep marker structure intact: only code bits change
        rc_h, px_h = run(bad, 1)
        rc_d, px_d = run(bad, 2)
        assert rc_h == rc_d, (t, rc_h, rc_d)
        if rc_h == 0:
            assert (px_h == px_d).all(), t
