"""No-GPU checks of the product library: it loads, exports every symbol declared in include/*.h,
its host-only entry points work, and compute entry points fail loudly (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return C.CDLL(T.GPU_SO)


def _declared():
    names = []
    for h in ("ultrahdr_api.h", "uhdr_b200.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        src = "\n".join(l for l in src.split("\n") if not l.lstrip().startswith("#"))
        names += re.findall(r"UHDR_EXTERN[^;(]*?\b(\w+)\s*\(", src)
    return sorted(set(names))


def test_exports_every_declared_symbol(lib):
    names = _declared()
    assert len(names) >= 43 + 15
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_reference_symbol_list_is_covered(lib):
    # every UHDR_EXTERN function of the reference's ultrahdr_api.h, one name per line
    names = set(open(os.path.join(ROOT, "tests", "golden", "reference_api_symbols.txt")).read().split())
    assert len(names) == 43
    assert not [n for n in names if not hasattr(lib, n)]


def test_lut_blob_builder_matches_oracle(lib, oracle_libs):
    lib.uhdr_b200_lut_blob_floats.restype = C.c_size_t
    n = lib.uhdr_b200_lut_blob_floats()
    blob = np.zeros(n, np.float32)
    assert lib.uhdr_b200_build_lut_blob(blob.ctypes.data_as(C.c_void_p)) == 0
    o = oracle_libs.Oracle()
    parts = ((0, 1024, 0), (1024, 4096, 1), (9216, 4096, 2), (13312, 65536, 3), (13312 + 65536, 65536, 4))
    for off, cnt, which in parts:
        assert (blob[off:off + cnt].view(np.uint32) == o.lut(which).view(np.uint32)).all(), which
    assert (blob[-256:] == (np.arange(256, dtype=np.float32) / np.float32(255.0))).all()


def test_encoder_state_machine_and_validation(lib):
    api = T.UhdrApi(lib)
    L = lib
    enc = C.c_void_p(L.uhdr_create_encoder())
    assert L.uhdr_enc_set_quality(enc, 101, A.BASE_IMG).error_code == 3
    assert L.uhdr_enc_set_quality(enc, 90, A.BASE_IMG).error_code == 0
    assert L.uhdr_enc_set_gainmap_scale_factor(enc, 0).error_code == 3
    assert L.uhdr_enc_set_gainmap_scale_factor(enc, 129).error_code == 3
    assert L.uhdr_enc_set_gainmap_gamma(enc, -1.0).error_code == 3
    assert L.uhdr_enc_set_min_max_content_boost(enc, 2.0, 1.0).error_code == 3
    assert L.uhdr_enc_set_raw_image(enc, None, A.HDR_IMG).error_code == 3
    w, h = 64, 32
    buf = T.make_p010(w, h)
    hdr, keep = A.p010_image(buf, w, h, A.CG_BT2100, A.CT_SRGB, A.CR_LIMITED)  # bad transfer for P010
    e = L.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG)
    assert e.error_code == 3 and b"color transfer" in e.detail
    hdr2, keep2 = A.p010_image(T.make_p010(63 + 1, 31 + 1), 63, 31, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    assert L.uhdr_enc_set_raw_image(enc, C.byref(hdr2), A.HDR_IMG).error_code == 3  # odd dims
    # encode with nothing set -> INVALID_OPERATION, then the handle has sailed
    assert L.uhdr_encode(enc).error_code == 5
    assert L.uhdr_enc_set_quality(enc, 80, A.BASE_IMG).error_code == 5
    L.uhdr_reset_encoder(enc)
    assert L.uhdr_enc_set_quality(enc, 80, A.BASE_IMG).error_code == 0
    assert L.uhdr_get_encoded_stream(enc) in (None,) or not L.uhdr_get_encoded_stream(enc)
    L.uhdr_release_encoder(enc)


def test_no_cpu_fallback(lib):
    """without a CUDA device every compute entry point must fail loudly"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    w, h = 64, 32
    hb = T.make_p010(w, h)
    sb = T.make_yuv420(w, h)
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    cfg = A.default_gm_config()
    gm = np.zeros((h, w, 3), np.uint8)
    gmi = A.raw_image(A.FMT_RGB888, -1, -1, -1, w, h, [gm], [w])
    md = A.GainmapMetadata()
    rc = lib.uhdr_b200_generate_gainmap(C.byref(sdr), C.byref(hdr), C.byref(cfg), C.byref(md), C.byref(gmi))
    assert rc != 0
    lib.uhdr_b200_last_error.restype = C.c_char_p
    assert b"CUDA" in lib.uhdr_b200_last_error()
    enc = C.c_void_p(lib.uhdr_create_encoder())
    lib.uhdr_enc_set_raw_image.restype = A.ErrorInfo
    e = lib.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG)
    assert e.error_code != 0 and b"CUDA" in e.detail
    lib.uhdr_release_encoder(enc)


def test_probe_reference_file_on_host(lib, oracle_libs):
    """uhdr_dec_probe / is_uhdr_image are host-only: run them on a file the reference wrote."""
    w, h = 256, 128
    hb = T.make_p010(w, h, "smooth")
    sb = T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    data = T.reference_file("capi/file_256x128_scale2", lambda: T.UhdrApi(oracle_libs.Ref().lib).encode(hdr, sdr, scale=2))
    buf = np.frombuffer(data, np.uint8).copy()
    assert lib.is_uhdr_image(buf.ctypes.data_as(C.c_void_p), len(data)) == 1
    assert lib.is_uhdr_image(buf.ctypes.data_as(C.c_void_p), 100) == 0
    api = T.UhdrApi(lib)
    dec = C.c_void_p(lib.uhdr_create_decoder())
    ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
    assert lib.uhdr_dec_set_image(dec, C.byref(ci)).error_code == 0
    assert lib.uhdr_dec_probe(dec).error_code == 0
    assert (lib.uhdr_dec_get_image_width(dec), lib.uhdr_dec_get_image_height(dec)) == (w, h)
    assert (lib.uhdr_dec_get_gainmap_width(dec), lib.uhdr_dec_get_gainmap_height(dec)) == (w // 2, h // 2)
    md = lib.uhdr_dec_get_gainmap_metadata(dec).contents

    def ref_md():
        # metadata the reference decoder reports for the same file
        ref = T.UhdrApi(oracle_libs.Ref().lib)
        rdec = C.c_void_p(ref.lib.uhdr_create_decoder())
        try:
            assert ref.lib.uhdr_dec_set_image(rdec, C.byref(ci)).error_code == 0
            assert ref.lib.uhdr_dec_probe(rdec).error_code == 0
            return bytes(ref.lib.uhdr_dec_get_gainmap_metadata(rdec).contents)
        finally:
            ref.lib.uhdr_release_decoder(rdec)
    assert T.same(bytes(md), T.from_reference("capi/probe_md_256x128_scale2", ref_md))
    assert lib.uhdr_dec_set_out_max_display_boost(dec, 2.0).error_code == 5  # probed -> not configurable
    lib.uhdr_release_decoder(dec)
