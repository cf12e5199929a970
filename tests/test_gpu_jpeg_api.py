"""GPU parity of the JPEG block stage and of the drop-in C API (uhdr_encode / uhdr_decode): the
coefficient blocks and the complete byte streams must equal the CPU checker's, and whole files must
be byte-identical to what the reference's own uhdr_encode writes (the reference build where oracle/_ref is
present, else the digests recorded from it, tests/golden/reference_digests.json)."""
import ctypes as C

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A

pytestmark = pytest.mark.gpu


def _img(fmt, w, h, kind, seed=3):
    rs = np.random.RandomState(seed)
    if fmt == A.FMT_YUV420:
        b = T.make_yuv420(w, h, kind, seed)
        img, keep = A.yuv420_image(b, w, h, 1)
        return img, (b, keep)
    if fmt == A.FMT_Y400:
        b = rs.randint(0, 256, w * h).astype(np.uint8) if kind == "noise" else \
            ((np.add.outer(np.arange(h) * 2, np.arange(w) * 3)) % 256).astype(np.uint8).ravel().copy()
        return A.raw_image(fmt, -1, -1, 1, w, h, [b], [w]), b
    if fmt == A.FMT_RGB888:
        b = rs.randint(0, 256, w * h * 3).astype(np.uint8) if kind == "noise" else \
            np.stack([(np.add.outer(np.arange(h) * k, np.arange(w) * (4 - k))) % 256 for k in (1, 2, 3)], -1).astype(np.uint8).ravel().copy()
        return A.raw_image(fmt, -1, -1, 1, w, h, [b], [w]), b
    if fmt == A.FMT_YUV444:
        b = rs.randint(0, 256, w * h * 3).astype(np.uint8)
        y, u, v = b[:w * h], b[w * h:2 * w * h], b[2 * w * h:]
        return A.raw_image(fmt, 1, 3, 1, w, h, [y, u, v], [w, w, w]), (b, y, u, v)
    raise ValueError(fmt)


SIZES = {A.FMT_YUV420: [(64, 48), (320, 240), (1280, 720)],
         A.FMT_Y400: [(64, 48), (320, 180), (960, 540), (72, 33)],
         A.FMT_RGB888: [(64, 48), (320, 180), (100, 61), (960, 540)],
         A.FMT_YUV444: [(64, 48), (96, 40)]}


@pytest.mark.parametrize("fmt", list(SIZES))
def test_forward_coefficients(gpu, oracle_libs, fmt):
    o = oracle_libs.Oracle().lib
    for (w, h) in SIZES[fmt]:
        for kind, q in (("noise", 95), ("smooth", 50), ("noise", 100), ("smooth", 7)):
            img, keep = _img(fmt, w, h, kind)
            f, ref = T.oracle_forward(o, img, q)
            got = T.gpu_jpeg_forward(gpu, img, q, f)
            for c in range(f.ncomp):
                assert (got[c] == ref[c]).all(), (fmt, w, h, kind, q, c, int((got[c] != ref[c]).sum()))


@pytest.mark.parametrize("fmt", list(SIZES))
def test_encode_stream_bytes(gpu, oracle_libs, fmt):
    o = oracle_libs.Oracle().lib
    icc = bytes(range(40))
    for (w, h) in SIZES[fmt]:
        for kind, q in (("noise", 95), ("smooth", 85)):
            img, keep = _img(fmt, w, h, kind)
            gm = fmt in (A.FMT_RGB888, A.FMT_Y400)
            ref = T.oracle_encode(o, img, q, icc, T.GM_COMMENT if gm else None)
            got = T.gpu_jpeg_encode(gpu, img, q, icc)
            assert got == ref, (fmt, w, h, kind, q, len(got), len(ref))


def test_decode_planes(gpu, oracle_libs):
    o = oracle_libs.Oracle().lib
    for fmt in (A.FMT_YUV420, A.FMT_Y400, A.FMT_RGB888):
        for (w, h) in SIZES[fmt]:
            img, keep = _img(fmt, w, h, "smooth")
            data = T.oracle_encode(o, img, 90)
            hd, planes = T.oracle_decode(o, data)
            f = hd.frame
            buf = np.zeros(w * h * 4 + 65536, np.uint8)
            out = A.raw_image(-1, -1, -1, -1, 0, 0, [buf], [0])
            cbuf = (C.c_uint8 * len(data)).from_buffer_copy(data)
            mode = 0 if fmt == A.FMT_YUV420 else 2
            rc = gpu.lib.uhdr_b200_jpeg_decode(cbuf, C.c_size_t(len(data)), mode, C.byref(out), C.c_size_t(buf.size))
            assert rc == 0, T.gpu_err(gpu)
            if f.ncomp == 1:
                got = buf[:w * h].reshape(h, w)
                assert (got == planes[0][:h, :w]).all()
            elif mode == 0:  # raw planes laid out like JpegDecoderHelper::getDecompressedImage
                assert out.fmt == A.FMT_YUV420 and out.stride[0] == w and out.stride[1] == w // 2
                off = 0
                for c, (pw, ph) in enumerate(((w, h), (w // 2, h // 2), (w // 2, h // 2))):
                    got = buf[off:off + pw * ph].reshape(ph, pw)
                    assert (got == planes[c][:ph, :pw]).all(), (w, h, c)
                    off += pw * ph
            else:  # DECODE_STREAM of a 3-component stream -> RGBA8888 through jdcolor.c
                assert out.fmt == A.FMT_RGBA8888
                got = buf[:w * h * 4].reshape(h, w, 4)
                r = np.zeros(1, np.uint8); g = np.zeros(1, np.uint8); b = np.zeros(1, np.uint8)
                rs = np.random.RandomState(0)
                for _ in range(200):
                    yy, xx = rs.randint(h), rs.randint(w)
                    o.jo_ycc_to_rgb(int(planes[0][yy, xx]), int(planes[1][yy, xx]), int(planes[2][yy, xx]),
                                    r.ctypes.data_as(C.c_void_p), g.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p))
                    assert tuple(got[yy, xx]) == (r[0], g[0], b[0], 255)


def _ref_api(oracle_libs):
    """the reference's C API, or None where its build is absent (recorded results stand in)"""
    return T.UhdrApi(oracle_libs.Ref().lib) if oracle_libs.have_ref() else None


def _ref_encoded(key, ref, mine, hdr, sdr, **opts):
    """a JPEG/R the reference wrote: live, or the product's file checked against the reference's digest"""
    return T.reference_file(key, lambda: ref.encode(hdr, sdr, **opts), mine=lambda: mine.encode(hdr, sdr, **opts))


def _frames(w, h, kind="smooth"):
    hb = T.make_p010(w, h, kind)
    sb = T.make_yuv420(w, h, kind)
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    return hdr, sdr, (hb, sb, k1, k2)


@pytest.mark.parametrize("w,h,kind", [(256, 128, "smooth"), (1280, 720, "smooth"), (640, 368, "noise")])
@pytest.mark.parametrize("opts", [{}, {"scale": 4, "multichannel": 0}, {"preset": A.USAGE_REALTIME, "quality": 80}])
def test_uhdr_encode_api1_file_bytes(gpu, oracle_libs, w, h, kind, opts):
    """uhdr_encode (API-1) through the drop-in C ABI == the reference's uhdr_encode, byte for byte."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, sdr, keep = _frames(w, h, kind)
    a = mine.encode(hdr, sdr, **opts)
    b = T.from_reference("jpeg_api/api1/%dx%d/%s/%s" % (w, h, kind, sorted(opts.items())), lambda: ref.encode(hdr, sdr, **opts))
    assert T.same(a, b), (len(a), b if isinstance(b, T.Recorded) else len(b))


def test_uhdr_decode_pixels(gpu, oracle_libs):
    """uhdr_decode of a reference-encoded file: RGBA half-float pixels, decoded gain map and metadata
    identical to the reference decoder's."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    for (w, h, opts) in ((640, 368, {}), (640, 368, {"scale": 4, "multichannel": 0}), (1280, 720, {"scale": 2})):
        hdr, sdr, keep = _frames(w, h)
        key = "jpeg_api/decode/%dx%d/%s" % (w, h, sorted(opts.items()))
        data = _ref_encoded(key + "/file", ref, mine, hdr, sdr, **opts)
        for fmt, ct in ((A.FMT_RGBAF16, A.CT_LINEAR), (A.FMT_RGBA1010102, A.CT_PQ)):
            got = mine.decode(data, fmt, ct)   # pixels, gain map, metadata, gamut
            want = T.from_reference(key + "/fmt%d_ct%d" % (fmt, ct), lambda: ref.decode(data, fmt, ct))
            assert T.same(got, want), (w, h, opts, fmt)


@pytest.mark.parametrize("w,h,kind", [(640, 368, "smooth"), (1280, 720, "noise")])
def test_uhdr_encode_api0_file_bytes(gpu, oracle_libs, w, h, kind):
    """API-0 (toneMap + one-pass gain map + both JPEGs) == the reference's file, byte for byte."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, sdr, keep = _frames(w, h, kind)
    for opts in ({}, {"multichannel": 0}, {"scale": 2}):
        want = T.from_reference("jpeg_api/api0/%dx%d/%s/%s" % (w, h, kind, sorted(opts.items())), lambda: ref.encode(hdr, None, **opts))
        assert T.same(mine.encode(hdr, None, **opts), want), opts


def _rgba_frames(w, h, hdr_kind):
    """packed intents: RGBA1010102 (PQ / HLG) or RGBA half float (linear) HDR + RGBA8888 SDR"""
    if hdr_kind == "f16":
        hb = T.make_rgbaf16(w, h)
        hdr = A.raw_image(A.FMT_RGBAF16, A.CG_BT2100, A.CT_LINEAR, A.CR_FULL, w, h, [hb], [w])
    else:
        hb = T.make_rgba1010102(w, h)
        hdr = A.raw_image(A.FMT_RGBA1010102, A.CG_BT2100, A.CT_PQ if hdr_kind == "pq" else A.CT_HLG, A.CR_FULL, w, h, [hb], [w])
    sb = T.make_rgba8888(w, h)
    sdr = A.raw_image(A.FMT_RGBA8888, A.CG_BT709, A.CT_SRGB, A.CR_FULL, w, h, [sb], [w])
    return hdr, sdr, (hb, sb)


@pytest.mark.parametrize("hdr_kind", ["pq", "hlg", "f16"])
def test_uhdr_encode_packed_intents_file_bytes(gpu, oracle_libs, hdr_kind):
    """RGBA1010102 / RGBA half-float HDR intents and the RGBA8888 SDR intent (convert_raw_input_to_ycbcr,
    4:4:4 base image): API-0 and API-1 files equal the reference's byte for byte."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    for (w, h) in ((320, 192), (648, 364)):
        hdr, sdr, keep = _rgba_frames(w, h, hdr_kind)
        key = "jpeg_api/packed/%s/%dx%d" % (hdr_kind, w, h)
        a, b = mine.encode(hdr, None), T.from_reference(key + "/api0", lambda: ref.encode(hdr, None))
        assert T.same(a, b), ("api0", hdr_kind, w, h, len(a))
        for opts in ({}, {"scale": 2, "multichannel": 0}):
            a = mine.encode(hdr, sdr, **opts)
            b = T.from_reference(key + "/api1/%s" % sorted(opts.items()), lambda: ref.encode(hdr, sdr, **opts))
            assert T.same(a, b), ("api1", hdr_kind, w, h, opts, len(a))


@pytest.mark.parametrize("subsampling", [2, 1, 0])
def test_decode_rgb_of_subsampled_streams(gpu, oracle_libs, subsampling):
    """DECODE_TO_RGB_CS of 4:2:0 / 4:2:2 / 4:4:4 streams written by a real libjpeg-turbo (Pillow):
    libjpeg's fancy chroma upsampling + colour conversion on the device == the CPU checker (which is
    pinned against Pillow's own decode in test_oracle_jpeg.py)."""
    PIL = pytest.importorskip("PIL.Image")
    import io
    o = oracle_libs.Oracle().lib
    for (w, h) in ((64, 48), (318, 237), (17, 9), (2, 2), (5, 3), (640, 361)):
        rs = np.random.RandomState(w + h)
        rgb = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        b = io.BytesIO()
        PIL.fromarray(rgb).save(b, "JPEG", quality=90, subsampling=subsampling)
        data = b.getvalue()
        hd, planes = T.oracle_decode(o, data)
        want = np.zeros((h, w, 4), np.uint8)
        pp = (C.c_void_p * 3)(*[p.ctypes.data for p in planes])
        assert o.jo_planes_to_rgba(C.byref(hd), pp, want.ctypes.data_as(C.c_void_p)) == 0
        for dec_mode in (1, 2):  # host and device entropy decoder
            prev = gpu.lib.uhdr_b200_set_entropy_decoder(dec_mode)
            try:
                buf = np.zeros(w * h * 4 + 65536, np.uint8)
                out = A.raw_image(-1, -1, -1, -1, 0, 0, [buf], [0])
                cbuf = (C.c_uint8 * len(data)).from_buffer_copy(data)
                rc = gpu.lib.uhdr_b200_jpeg_decode(cbuf, C.c_size_t(len(data)), 1, C.byref(out), C.c_size_t(buf.size))
            finally:
                gpu.lib.uhdr_b200_set_entropy_decoder(prev)
            assert rc == 0, T.gpu_err(gpu)
            assert out.fmt == A.FMT_RGBA8888
            got = buf[:w * h * 4].reshape(h, w, 4)
            assert (got == want).all(), (w, h, subsampling, dec_mode, int((got != want).sum()))


def test_uhdr_decode_sdr_output(gpu, oracle_libs):
    """uhdr_decode with UHDR_CT_SRGB / RGBA8888: the base image through libjpeg's RGB path, gain map and
    metadata still available -- identical to the reference decoder."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    for (w, h, opts) in ((640, 368, {}), (322, 182, {"scale": 2, "multichannel": 0})):
        hdr, sdr, keep = _frames(w, h)
        key = "jpeg_api/decode_sdr/%dx%d/%s" % (w, h, sorted(opts.items()))
        data = _ref_encoded(key + "/file", ref, mine, hdr, sdr, **opts)
        got = mine.decode(data, A.FMT_RGBA8888, A.CT_SRGB)
        want = T.from_reference(key + "/decoded", lambda: ref.decode(data, A.FMT_RGBA8888, A.CT_SRGB))
        assert T.same(got, want), (w, h, opts)


def test_uhdr_decode_444_base(gpu, oracle_libs):
    """files written from an RGBA8888 SDR intent carry a 4:4:4 base image: decode (half float, PQ
    1010102 and SDR outputs) == the reference decoder."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, sdr, keep = _rgba_frames(328, 200, "pq")
    for opts in ({}, {"scale": 2}):
        key = "jpeg_api/decode_444/328x200/%s" % sorted(opts.items())
        data = _ref_encoded(key + "/file", ref, mine, hdr, sdr, **opts)
        for fmt, ct in ((A.FMT_RGBAF16, A.CT_LINEAR), (A.FMT_RGBA1010102, A.CT_PQ), (A.FMT_RGBA1010102, A.CT_HLG), (A.FMT_RGBA8888, A.CT_SRGB)):
            got = mine.decode(data, fmt, ct)
            want = T.from_reference(key + "/fmt%d_ct%d" % (fmt, ct), lambda: ref.decode(data, fmt, ct))
            assert T.same(got, want), (opts, fmt, ct)


def test_encode_batch_matches_single_encodes(gpu, oracle_libs):
    """uhdr_b200_encode_batch (N frames pipelined over several streams / worker threads) returns,
    frame by frame, the bytes uhdr_encode returns for the same inputs."""
    lib = gpu.lib
    mine = T.UhdrApi(lib)
    w, h, n = 640, 368, 7
    keeps, hdrs, sdrs = [], (A.RawImage * n)(), (A.RawImage * n)()
    singles = []
    for i in range(n):
        hb = T.make_p010(w, h, "smooth", seed=100 + i)
        sb = T.make_yuv420(w, h, "smooth", seed=200 + i)
        hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
        sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
        keeps.append((hb, sb, k1, k2))
        hdrs[i], sdrs[i] = hdr, sdr
        singles.append(mine.encode(hdr, sdr))
    cap = w * h * 6 + 65536
    bufs = [np.zeros(cap, np.uint8) for _ in range(n)]
    outs = (A.CompressedImage * n)()
    for i in range(n):
        outs[i] = A.CompressedImage(bufs[i].ctypes.data, 0, cap, -1, -1, -1)
    cfg = A.default_gm_config()
    for streams in (1, 3):
        rc = lib.uhdr_b200_encode_batch(n, hdrs, sdrs, C.byref(cfg), 95, outs, streams)
        assert rc == 0, T.gpu_err(gpu)
        for i in range(n):
            got = bytes(bufs[i][:outs[i].data_sz])
            assert got == singles[i], (streams, i, len(got), len(singles[i]))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,kind", [(256, 128, "smooth"), (648, 364, "noise"), (1920, 1080, "smooth")])
def test_uhdr_encode_api2_api3_file_bytes(gpu, oracle_libs, w, h, kind):
    """Encode API-2 (raw hdr + raw sdr + compressed sdr) and API-3 (raw hdr + compressed sdr: the JPEG is
    decoded on the device, the gain map computed against it with BT.601 luma): files equal the reference's."""
    PIL = pytest.importorskip("PIL.Image")
    import io
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, sdr, keep = _frames(w, h, kind)
    # compressed sdr intents: the reference's own base image (4:2:0, with ICC) and a Pillow file (4:2:0 / 4:4:4, no ICC)
    from test_probe_cpu import _probe
    key = "jpeg_api/api2_api3/%dx%d/%s" % (w, h, kind)
    base_ref = T.reference_file(key + "/base_image", lambda: _probe(ref.lib, ref.encode(hdr, sdr))["base_image"],
                                mine=lambda: _probe(gpu.lib, mine.encode(hdr, sdr))["base_image"])
    rgb = np.random.RandomState(5).randint(0, 256, (h, w, 3)).astype(np.uint8)
    pil = {}
    for ss in (2, 0):
        b = io.BytesIO()
        PIL.fromarray(rgb).save(b, "JPEG", quality=90, subsampling=ss)
        pil[ss] = b.getvalue()
    cases = [("api2", base_ref, sdr, -1, {}), ("api2", base_ref, sdr, -1, {"scale": 2, "multichannel": 0}),
             ("api3", base_ref, None, -1, {}), ("api3", base_ref, None, A.CG_BT709, {"multichannel": 0}),
             ("api3", pil[2], None, A.CG_P3, {}), ("api3", pil[0], None, A.CG_BT709, {"scale": 2}),
             ("api3", pil[2], None, -1, {}),           # no ICC and no gamut: error in both
             ("api3", base_ref, None, A.CG_BT2100, {})]  # configured gamut contradicts the ICC: error in both
    for i, (name, jpg, raw, cg, opts) in enumerate(cases):
        a = mine.encode_with_compressed_sdr(hdr, jpg, raw, cg, **opts)   # the file, or the error code
        b = T.from_reference(key + "/case%d" % i, lambda: ref.encode_with_compressed_sdr(hdr, jpg, raw, cg, **opts))
        assert T.same(a, b), (name, cg, opts, a if isinstance(a, int) else len(a))
