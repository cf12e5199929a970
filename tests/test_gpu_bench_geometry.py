"""Parity at the geometries the benchmark and the reference's own benchmark use (VERDICT r1, weak #3):
whole files at 3840x2160 on bench.py's frame generator (API-1 and API-0), re-armed encodes of resident
inputs, 7680x4320 uhdr_decode, 1920x1080 / 4080x3072 (benchmark/benchmark_test.cpp:55-72 of the
reference; both have MCU rows / columns that reach past the block grid), config 1 on the reference's
real 720p fixtures, and a 4:2:2 base image through applyGainMap.  Without oracle/_ref, the digests
recorded from the reference build (tests/golden/reference_digests.json) stand in for its results."""
import ctypes as C
import io

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A

pytestmark = pytest.mark.gpu


def _bench_frame(w, h, idx):
    import bench
    p, y = bench.make_frame(w, h, idx)
    hdr, sdr, keep = bench.frame_descs(p, y, w, h)
    return hdr, sdr, (p, y, keep)


def _ref_api(oracle_libs):
    """the reference's C API, or None where its build is absent (recorded results stand in)"""
    return T.UhdrApi(oracle_libs.Ref().lib) if oracle_libs.have_ref() else None


def test_4k_api1_file_and_rearmed_encodes(gpu, oracle_libs):
    """uhdr_encode at the headline geometry == the reference's file; encoding the same resident inputs
    again (uhdr_b200_enc_rearm, what bench.py's `value` arm does) returns the same bytes every time."""
    ref = _ref_api(oracle_libs)
    lib = gpu.lib
    T.UhdrApi(lib)
    hdr, sdr, keep = _bench_frame(3840, 2160, 3)
    want = T.from_reference("bench_geometry/4k_api1", lambda: ref.encode(hdr, sdr))
    enc = C.c_void_p(lib.uhdr_create_encoder())
    try:
        assert lib.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG).error_code == 0
        assert lib.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG).error_code == 0
        for it in range(3):
            e = lib.uhdr_encode(enc)
            assert e.error_code == 0, e.detail
            o = lib.uhdr_get_encoded_stream(enc).contents
            got = C.string_at(o.data, o.data_sz)
            assert T.same(got, want), (it, len(got))
            assert lib.uhdr_b200_enc_rearm(enc) == 0
    finally:
        lib.uhdr_release_encoder(enc)


def test_4k_api0_file(gpu, oracle_libs):
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, _sdr, keep = _bench_frame(3840, 2160, 5)
    assert T.same(mine.encode(hdr, None), T.from_reference("bench_geometry/4k_api0", lambda: ref.encode(hdr, None)))


@pytest.mark.parametrize("w,h", [(1920, 1080), (4080, 3072)])
def test_reference_benchmark_sizes(gpu, oracle_libs, w, h):
    """API-1 and API-0 files at the sizes of the reference's own benchmark.  1080 = 67.5 MCU rows and
    4080 = 255 MCU columns: libjpeg's dummy-block rule and the helper's chroma padding are in play."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, sdr, keep = _bench_frame(w, h, 9)
    key = "bench_geometry/%dx%d" % (w, h)
    a = mine.encode(hdr, sdr)
    b = T.reference_file(key + "/api1", lambda: ref.encode(hdr, sdr), mine=lambda: a)
    api0 = T.from_reference(key + "/api0_single_channel", lambda: ref.encode(hdr, None, multichannel=0))
    assert T.same(mine.encode(hdr, None, multichannel=0), api0)
    got = mine.decode(b)
    assert T.same(got, T.from_reference(key + "/decoded", lambda: ref.decode(b)))


def test_8k_uhdr_decode(gpu, oracle_libs):
    """config 3: uhdr_decode of a 7680x4320 JPEG/R to RGBA half float, device entropy decoder: pixels,
    gain map, metadata and gamut == the reference decoder's."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    hdr, sdr, keep = _bench_frame(7680, 4320, 7)
    data = mine.encode(hdr, sdr)
    assert T.same(data, T.from_reference("bench_geometry/8k_api1", lambda: ref.encode(hdr, sdr)))
    st0, st1 = (C.c_ulonglong * 3)(), (C.c_ulonglong * 3)()
    gpu.lib.uhdr_b200_entropy_decoder_stats.restype = None
    gpu.lib.uhdr_b200_entropy_decoder_stats(st0)
    pa, ga, ma, cga = mine.decode(data)
    gpu.lib.uhdr_b200_entropy_decoder_stats(st1)
    assert st1[0] - st0[0] == 2 and st1[1] == st0[1], "both scans must go through the device entropy decoder"
    assert T.same((pa, ga, ma, cga), T.from_reference("bench_geometry/8k_decoded", lambda: ref.decode(data)))


def test_config1_real_fixtures(gpu, oracle_libs):
    """BASELINE config 1: the reference's own 1280x720 fixtures (stored in tests/golden), ultrahdr_app's
    defaults: hdr P3 HLG limited, sdr BT.709."""
    ref = _ref_api(oracle_libs)
    mine = T.UhdrApi(gpu.lib)
    w, h = 1280, 720
    p, y = T.load_fixture_720p()
    p = p[:w * h * 3 // 2].copy()
    y = y[:w * h * 3 // 2].copy()
    hdr, k1 = A.p010_image(p, w, h, A.CG_P3, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(y, w, h, A.CG_BT709)
    a = mine.encode(hdr, sdr)
    b = T.reference_file("bench_geometry/config1/api1", lambda: ref.encode(hdr, sdr), mine=lambda: a)
    assert T.same(mine.encode(hdr, None), T.from_reference("bench_geometry/config1/api0", lambda: ref.encode(hdr, None)))
    for fmt, ct in ((A.FMT_RGBAF16, A.CT_LINEAR), (A.FMT_RGBA1010102, A.CT_HLG), (A.FMT_RGBA1010102, A.CT_PQ)):
        got = mine.decode(b, fmt, ct)
        want = T.from_reference("bench_geometry/config1/fmt%d_ct%d" % (fmt, ct), lambda: ref.decode(b, fmt, ct))
        assert T.same(got, want), (fmt, ct)


@pytest.mark.parametrize("subsampling,name", [(1, "4:2:2"), (0, "4:4:4"), (2, "4:2:0")])
def test_apply_on_subsampled_base(gpu, oracle_libs, subsampling, name):
    """applyGainMap with a 4:2:2 (and 4:4:4 / 4:2:0) base image: the base JPEG comes from a real
    libjpeg-turbo (Pillow), the stage result must equal the reference's applyGainMap on the same planes."""
    PIL = pytest.importorskip("PIL.Image")
    chk = oracle_libs.Ref() if oracle_libs.have_ref() else None
    w, h = 322, 182
    rs = np.random.RandomState(11)
    yy, xx = np.mgrid[0:h, 0:w]
    rgb = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) % 256)], -1).astype(np.uint8)
    b = io.BytesIO()
    PIL.fromarray(rgb).save(b, "JPEG", quality=92, subsampling=subsampling)
    data = b.getvalue()
    # decode to raw planes with the product (uhdr_b200_jpeg_decode mode 0 = DECODE_TO_YCBCR_CS)
    buf = np.zeros(w * h * 4 + 65536, np.uint8)
    out = A.raw_image(-1, -1, -1, -1, 0, 0, [buf], [0])
    cbuf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    assert gpu.lib.uhdr_b200_jpeg_decode(cbuf, C.c_size_t(len(data)), 0, C.byref(out), C.c_size_t(buf.size)) == 0, T.gpu_err(gpu)
    assert out.fmt == {1: A.FMT_YUV422, 0: A.FMT_YUV444, 2: A.FMT_YUV420}[subsampling]
    out.cg = A.CG_BT709
    out.ct = A.CT_SRGB
    out.range = A.CR_FULL
    gm = rs.randint(0, 256, (h // 2, w // 2, 3)).astype(np.uint8)
    gi = T.gm_image(gm, A.CG_P3)
    md = A.GainmapMetadata()
    for i in range(3):
        md.max_content_boost[i], md.min_content_boost[i], md.gamma[i] = 6.0 + i, 0.8, 1.0
        md.offset_sdr[i] = md.offset_hdr[i] = 1e-7
    md.hdr_capacity_min, md.hdr_capacity_max, md.use_base_cg = 1.0, 6.0, 1
    for ct in (A.CT_LINEAR, A.CT_PQ, A.CT_HLG):
        a = gpu.apply(out, gi, md, ct)
        bb = T.from_reference("bench_geometry/apply_subsampled/%s/ct%d" % (name, ct), lambda: chk.apply(out, gi, md, ct))
        assert T.same(a, bb), (name, ct)
