"""GPU parity of the four per-pixel stages against the CPU checker (reference build when present,
else the C restatement), called through the C ABI with host buffers.  Bit-exact bar for the packed
integer outputs and for the RGBA-F16 / metadata floats (tolerance 0 ULP is asserted; the tests that
involve float powf with a continuous argument state their own bound)."""
import ctypes as C
import itertools

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A

pytestmark = pytest.mark.gpu
W, H = 96, 64


def _hdr(kind, fmt, cg, ct, w=W, h=H):
    if fmt == "p010":
        b = T.make_p010(w, h, kind)
        img, keep = A.p010_image(b, w, h, cg, ct, A.CR_LIMITED)
    elif fmt == "p010full":
        b = T.make_p010(w, h, kind, limited=False)
        img, keep = A.p010_image(b, w, h, cg, ct, A.CR_FULL)
    elif fmt == "1010102":
        b = T.make_rgba1010102(w, h)
        img, keep = A.raw_image(A.FMT_RGBA1010102, cg, ct, A.CR_FULL, w, h, [b], [w]), b
    else:
        b = T.make_rgbaf16(w, h)
        img, keep = A.raw_image(A.FMT_RGBAF16, cg, A.CT_LINEAR, A.CR_FULL, w, h, [b], [w]), b
    return img, (b, keep)


def _sdr(kind, cg, w=W, h=H):
    b = T.make_yuv420(w, h, kind)
    img, keep = A.yuv420_image(b, w, h, cg)
    return img, (b, keep)


GEN_CASES = list(itertools.product(["noise", "smooth", "black"], [A.CT_HLG, A.CT_PQ], [0, 1, 2],
                                   [0, 1, 2], [0, 1], [1, 2, 4], [0, 1]))


def test_generate_matrix(gpu, checker):
    bad = []
    for kind, hct, hcg, scg, multi, scale, preset in GEN_CASES:
        hdr, k1 = _hdr(kind, "p010", hcg, hct)
        sdr, k2 = _sdr(kind, scg)
        cfg = A.default_gm_config(scale_factor=scale, multichannel=multi, preset=preset)
        g1, m1 = gpu.generate(sdr, hdr, cfg)
        g2, m2 = checker.generate(sdr, hdr, cfg)
        if not ((g1 == g2).all() and T.md_equal(m1, m2)):
            bad.append((kind, hct, hcg, scg, multi, scale, preset, int((g1 != g2).sum())))
    assert not bad, bad[:10]


def test_generate_srgb_transfer_leg(gpu, checker):
    """config 5's sRGB leg: an sRGB-transfer P010 "hdr" intent is refused by uhdr_enc_set_raw_image but is a
    valid JpegR::generateGainMap input (getInverseOetfFn, gainmapmath.cpp:1175-1180)."""
    bad = []
    for hcg, scg, multi, scale, preset in itertools.product([0, 1, 2], [0, 2], [0, 1], [1, 2, 4], [0, 1]):
        hdr, k1 = _hdr("noise", "p010", hcg, A.CT_SRGB)
        sdr, k2 = _sdr("noise", scg)
        cfg = A.default_gm_config(scale_factor=scale, multichannel=multi, preset=preset)
        g1, m1 = gpu.generate(sdr, hdr, cfg)
        g2, m2 = checker.generate(sdr, hdr, cfg)
        if not ((g1 == g2).all() and T.md_equal(m1, m2)):
            bad.append((hcg, scg, multi, scale, preset, int((g1 != g2).sum())))
    assert not bad, bad[:10]


@pytest.mark.parametrize("fmt,ct", [("p010full", A.CT_HLG), ("1010102", A.CT_PQ), ("1010102", A.CT_HLG),
                                    ("f16", A.CT_LINEAR)])
@pytest.mark.parametrize("multi,preset", [(1, 1), (1, 0), (0, 1), (0, 0)])
def test_generate_formats(gpu, checker, fmt, ct, multi, preset):
    hdr, k1 = _hdr("noise", fmt, 2, ct)
    sdr, k2 = _sdr("noise", 0)
    for extra in ({}, {"use_luminance": 0}, {"sdr_is_601": 1}, {"scale_factor": 2}):
        cfg = A.default_gm_config(multichannel=multi, preset=preset, **extra)
        g1, m1 = gpu.generate(sdr, hdr, cfg)
        g2, m2 = checker.generate(sdr, hdr, cfg)
        assert (g1 == g2).all(), (extra, int((g1 != g2).sum()))
        assert T.md_equal(m1, m2), (m1.as_dict(), m2.as_dict())


def test_generate_rgba8888_sdr_and_boost_hints(gpu, checker):
    hdr, k1 = _hdr("noise", "p010", 2, A.CT_HLG)
    sb = T.make_rgba8888(W, H)
    sdr = A.raw_image(A.FMT_RGBA8888, 0, A.CT_SRGB, A.CR_FULL, W, H, [sb], [W])
    for kw in ({}, {"min_content_boost": 0.5, "max_content_boost": 6.0}, {"target_disp_peak_nits": 1600.0},
               {"preset": 0, "target_disp_peak_nits": 800.0}):
        cfg = A.default_gm_config(**kw)
        g1, m1 = gpu.generate(sdr, hdr, cfg)
        g2, m2 = checker.generate(sdr, hdr, cfg)
        assert (g1 == g2).all() and T.md_equal(m1, m2), kw


def test_generate_fast_path_hints_and_degenerate_ranges(gpu, checker):
    """The quotient-plane two-pass path (P010 + YUV420) with content-boost hints (they clamp min / max after the
    extremes were found, which makes the affine range small and many values saturate), with constant images (range
    forced to 0.1 by the |max - min| < eps rule), with an all-dark SDR image (only the capped class exists), at
    scales 1 / 4 and both channel counts."""
    bad = []
    for kind, scale, multi in itertools.product(["noise", "smooth", "black", "white"], [1, 4], [0, 1]):
        hdr, k1 = _hdr(kind, "p010", 2, A.CT_PQ)
        sdr, k2 = _sdr(kind, 0)
        for kw in ({}, {"min_content_boost": 0.5, "max_content_boost": 6.0}, {"min_content_boost": 1.0, "max_content_boost": 1.25},
                   {"max_content_boost": 0.9, "min_content_boost": 0.8}, {"target_disp_peak_nits": 1600.0}):
            cfg = A.default_gm_config(scale_factor=scale, multichannel=multi, **kw)
            g1, m1 = gpu.generate(sdr, hdr, cfg)
            g2, m2 = checker.generate(sdr, hdr, cfg)
            if not ((g1 == g2).all() and T.md_equal(m1, m2)):
                bad.append((kind, scale, multi, kw, int((g1 != g2).sum())))
    # dark HDR over bright SDR and the reverse: every gain at one end
    for hk, sk in (("black", "white"), ("white", "black")):
        hdr, k1 = _hdr(hk, "p010", 2, A.CT_HLG)
        sdr, k2 = _sdr(sk, 0)
        g1, m1 = gpu.generate(sdr, hdr)
        g2, m2 = checker.generate(sdr, hdr)
        if not ((g1 == g2).all() and T.md_equal(m1, m2)):
            bad.append((hk, sk, int((g1 != g2).sum())))
    assert not bad, bad[:8]


def _map_for(gpu_or_chk, kind, multi, scale):
    hdr, k1 = _hdr(kind, "p010", 2, A.CT_HLG)
    sdr, k2 = _sdr(kind, 0)
    cfg = A.default_gm_config(scale_factor=scale, multichannel=multi)
    g, m = gpu_or_chk.generate(sdr, hdr, cfg)
    return sdr, k2, g, m


@pytest.mark.parametrize("out_ct", [A.CT_LINEAR, A.CT_PQ])
def test_apply_matrix(gpu, checker, out_ct):
    bad = []
    for kind, (multi, scale) in itertools.product(["noise", "smooth"], [(1, 1), (0, 1), (1, 4), (0, 4), (1, 2)]):
        sdr, keep, g, m = _map_for(checker, kind, multi, scale)
        variants = [g] if not multi else [g, np.concatenate([g, np.full(g.shape[:2] + (1,), 255, np.uint8)], -1)]
        for gm in variants:
            gm = np.ascontiguousarray(gm)
            for gcg, boost in itertools.product([-1, 0, 1, 2], [A.FLT_MAX, 2.5]):
                gi = T.gm_image(gm, gcg)
                a = gpu.apply(sdr, gi, m, out_ct, boost)
                b = checker.apply(sdr, gi, m, out_ct, boost)
                if not (a == b).all():
                    bad.append((kind, multi, scale, gm.shape[2], gcg, boost, int((a != b).sum())))
    assert not bad, bad[:10]


def test_apply_hlg_output(gpu, checker):
    """HLG output goes through float powf(x, 1/1.2f) with a continuous argument; the device runs
    glibc's powf operation for operation (powf_glibc.cuh), so the packed pixels are bit-exact."""
    for multi, scale in ((1, 1), (0, 4)):
        sdr, keep, g, m = _map_for(checker, "noise", multi, scale)
        for gcg in (2, 0):
            gi = T.gm_image(g, gcg)
            a = gpu.apply(sdr, gi, m, A.CT_HLG)
            b = checker.apply(sdr, gi, m, A.CT_HLG)
            assert (a == b).all(), (multi, scale, gcg, int((a != b).sum()))


def test_apply_non_integer_scale(gpu, checker):
    sdr, keep, g, m = _map_for(checker, "noise", 1, 1)
    for ch in (1, 3):
        gm = np.ascontiguousarray(g[:43, :64, :ch])
        gi = T.gm_image(gm, 2)
        for ct in (A.CT_LINEAR, A.CT_PQ):
            a = gpu.apply(sdr, gi, m, ct)
            b = checker.apply(sdr, gi, m, ct)
            assert (a == b).all(), (ch, ct, int((a != b).sum()))


def test_apply_gamma_metadata(gpu, checker):
    """gamma != 1 routes through pow(double) on both sides (GainLUT::getGainFactor)."""
    hdr, k1 = _hdr("noise", "p010", 2, A.CT_HLG)
    sdr, k2 = _sdr("noise", 0)
    cfg = A.default_gm_config(gamma=2.2)
    g, m = checker.generate(sdr, hdr, cfg)
    gi = T.gm_image(g, 2)
    a = gpu.apply(sdr, gi, m, A.CT_LINEAR)
    b = checker.apply(sdr, gi, m, A.CT_LINEAR)
    # device pow() and glibc pow() are both <1-2 ulp in double; index flips need a tie
    assert (a != b).sum() <= 1e-5 * a.size


def test_tonemap(gpu, checker):
    """toneMap's srgbOetf is float powf on a continuous argument: evaluated as glibc does
    (powf_glibc.cuh), so the packed 8-bit planes are bit-exact."""
    for kind, hct, hcg in itertools.product(["noise", "smooth", "white", "black"], [A.CT_HLG, A.CT_PQ], [0, 1, 2]):
        hdr, k = _hdr(kind, "p010", hcg, hct)
        a, _ = gpu.tonemap(hdr)
        b, _ = checker.tonemap(hdr)
        assert (a == b).all(), (kind, hct, hcg, int((a != b).sum()))
    hdr, k = _hdr("noise", "p010full", 2, A.CT_HLG)
    assert (gpu.tonemap(hdr)[0] == checker.tonemap(hdr)[0]).all()


def test_tonemap_rgba(gpu, checker):
    for fmt, ct in (("1010102", A.CT_PQ), ("1010102", A.CT_HLG), ("f16", A.CT_LINEAR)):
        hdr, k = _hdr("noise", fmt, 2, ct)
        a, _ = gpu.tonemap(hdr)
        b, _ = checker.tonemap(hdr)
        assert (a == b).all(), (fmt, ct)


def test_tonemap_4k(gpu, checker):
    """config 2 geometry"""
    w, h = 3840, 2160
    hb = T.make_p010(w, h, "noise")
    hdr, k = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    assert (gpu.tonemap(hdr)[0] == checker.tonemap(hdr)[0]).all()


def test_device_powf_equals_libm(gpu, oracle_libs):
    """glibc powf restated on the device: identical bits on dense samples of [0, 1] for the
    exponents the hot path uses (1/2.4, 1/1.2) and a gain-map gamma."""
    import ctypes as C
    o = oracle_libs.Oracle().lib
    o.uo_powf_vec.argtypes = [C.c_void_p, C.c_float, C.c_void_p, C.c_size_t]
    gpu.lib.uhdr_b200_probe_powf.argtypes = [C.c_void_p, C.c_float, C.c_void_p, C.c_int]
    rs = np.random.RandomState(5)
    x = np.concatenate([rs.uniform(0, 1, 4_000_000), np.exp(rs.uniform(np.log(1e-45), 0, 1_000_000)),
                        np.arange(0, 65536) / 65535.0, [0.0, 1.0, 1e-45, 1.1754944e-38, 0.0031308, 0.5]]).astype(np.float32)
    x = np.ascontiguousarray(x)
    for y in (1.0 / 2.4, 1.0 / 1.2, 2.2, 1.2):
        yf = float(np.float32(np.float32(1.0) / np.float32(2.4))) if abs(y - 1 / 2.4) < 1e-9 else \
            float(np.float32(np.float32(1.0) / np.float32(1.2))) if abs(y - 1 / 1.2) < 1e-9 else float(np.float32(y))
        want = np.zeros_like(x)
        got = np.zeros_like(x)
        o.uo_powf_vec(x.ctypes.data, yf, want.ctypes.data, x.size)
        assert gpu.lib.uhdr_b200_probe_powf(x.ctypes.data, yf, got.ctypes.data, x.size) == 0
        bad = got.view(np.uint32) != want.view(np.uint32)
        assert bad.sum() == 0, (y, int(bad.sum()), x[bad][:4], got[bad][:4], want[bad][:4])


def test_generate_onepass_gamma(gpu, checker):
    """REALTIME preset with gamma != 1: encodeGain's powf(gain_normalized, gamma)"""
    hdr, k1 = _hdr("noise", "p010", 2, A.CT_HLG)
    sdr, k2 = _sdr("noise", 0)
    for gamma in (2.2, 0.7):
        cfg = A.default_gm_config(preset=0, gamma=gamma)
        g1, m1 = gpu.generate(sdr, hdr, cfg)
        g2, m2 = checker.generate(sdr, hdr, cfg)
        assert (g1 == g2).all() and T.md_equal(m1, m2), gamma


def test_convert_yuv(gpu, checker):
    for s, d in itertools.permutations([0, 1, 2], 2):
        sb = T.make_yuv420(W, H, "noise")
        a = gpu.convert_yuv(sb, W, H, s, d)
        b = checker.convert_yuv(sb, W, H, s, d)
        assert (a == b).all(), (s, d)


def test_convert_yuv_444_and_unsupported_formats(gpu, checker):
    """convertYuv at stage level on a 4:4:4 image (transformYuv444, jpegr.cpp:504-507) for all six gamut pairs, and the
    reference's refusal of every other layout (:508-514), e.g. 4:2:2."""
    rs = np.random.RandomState(5)
    w, h = 98, 54
    for s, d in itertools.permutations([0, 1, 2], 2):
        outs = []
        for impl in (gpu, checker):
            planes = [rs_plane.copy() for rs_plane in _planes444(w, h)]
            img = A.raw_image(A.FMT_YUV444, s, A.CT_SRGB, A.CR_FULL, w, h, planes, [w, w, w])
            assert impl.f("convert_yuv")(C.byref(img), s, d) == 0
            outs.append(np.stack(planes))
        assert (outs[0] == outs[1]).all(), (s, d, int((outs[0] != outs[1]).sum()))
    planes = [rs.randint(0, 256, (h, w)).astype(np.uint8), rs.randint(0, 256, (h, w // 2)).astype(np.uint8),
              rs.randint(0, 256, (h, w // 2)).astype(np.uint8)]
    for impl in (gpu, checker):
        img = A.raw_image(A.FMT_YUV422, 0, A.CT_SRGB, A.CR_FULL, w, h, planes, [w, w // 2, w // 2])
        assert impl.f("convert_yuv")(C.byref(img), 0, 1) != 0


def _planes444(w, h):
    rs = np.random.RandomState(17)
    return [rs.randint(0, 256, (h, w)).astype(np.uint8) for _ in range(3)]


def test_lut_blob_matches_checker(gpu, checker):
    n = gpu.lib.uhdr_b200_lut_blob_floats
    n.restype = np.ctypeslib.ctypes.c_size_t
    blob = np.zeros(n(), np.float32)
    assert gpu.lib.uhdr_b200_get_lut_blob(blob.ctypes.data_as(np.ctypeslib.ctypes.c_void_p)) == 0
    off = 0
    srgb, hlginv = blob[0:1024], blob[1024:5120]
    pqinv = blob[9216:13312]
    hlgo = blob[13312:13312 + 65536]
    pqo = blob[13312 + 65536:13312 + 131072]
    for mine, which in ((srgb, 0), (hlginv, 1), (pqinv, 2), (hlgo, 3), (pqo, 4)):
        ref = checker.lut(which)
        assert (mine.view(np.uint32) == ref.view(np.uint32)).all(), which


@pytest.mark.parametrize("w,h", [(1280, 720), (3840, 2160)])
def test_api1_stages_full_size(gpu, checker, w, h):
    """config 1 / config 4 geometry on synthetic frames: default API-1 settings."""
    hb = T.make_p010(w, h, "noise")
    sb = T.make_yuv420(w, h, "noise")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    g1, m1 = gpu.generate(sdr, hdr)
    g2, m2 = checker.generate(sdr, hdr)
    assert T.md_equal(m1, m2), (m1.as_dict(), m2.as_dict())
    assert (g1 == g2).all(), int((g1 != g2).sum())
    a = gpu.convert_yuv(sb, w, h, 0, 1)
    b = checker.convert_yuv(sb, w, h, 0, 1)
    assert (a == b).all()


@pytest.mark.parametrize("w,h,scale,multi,preset", [(3840, 2160, 4, 0, 0), (3840, 2160, 4, 0, 1), (3840, 2160, 4, 1, 1),
                                                    (1920, 1080, 2, 1, 1), (1920, 1080, 2, 0, 0), (1284, 724, 4, 0, 1)])
def test_generate_scaled_full_size(gpu, checker, w, h, scale, multi, preset):
    """JpegR's own defaults (map scale 4, one channel, ultrahdrcommon.h:450-457) and scale 2 at full
    size: k_gainmap_scaled against the reference's samplePixels path, bit exact."""
    hb = T.make_p010(w, h, "noise")
    sb = T.make_yuv420(w, h, "noise")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    cfg = A.default_gm_config(scale_factor=scale, multichannel=multi, preset=preset)
    g1, m1 = gpu.generate(sdr, hdr, cfg)
    g2, m2 = checker.generate(sdr, hdr, cfg)
    assert g1.shape == g2.shape == (h // scale, w // scale, 3 if multi else 1) or g1.shape == g2.shape
    assert T.md_equal(m1, m2), (m1.as_dict(), m2.as_dict())
    assert (g1 == g2).all(), int((g1 != g2).sum())


def test_fast_pow_error_bound(gpu):
    """toneMap's screen (tonemap_fast.cu) trusts ex2.approx(lg2.approx(e) / 2.4) to within 3e-7 of the exact powf
    restatement for every float e in (0.0031308, 1]: all of them are compared on the device, and the worst case must
    leave a factor 2."""
    import struct
    lib = gpu.lib
    first = struct.unpack("<I", struct.pack("<f", 0.0031308))[0]
    last = struct.unpack("<I", struct.pack("<f", 1.0))[0]
    worst = C.c_float(-1.0)
    assert lib.uhdr_b200_probe_pow_fast(C.c_uint(first), C.c_uint(last - first + 1), C.byref(worst)) == 0, T.gpu_err(gpu)
    assert 0.0 < worst.value <= 1.5e-7, worst.value


def test_tonemap_redoes_only_groups_near_a_rounding_boundary(gpu, checker):
    lib = gpu.lib

    def stats():
        st = (C.c_ulonglong * 2)()
        lib.uhdr_b200_tonemap_stats(st)
        return st[0], st[1]
    w, h = 1280, 720
    hb = T.make_p010(w, h, "noise")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    g0, e0 = stats()
    a = gpu.tonemap(hdr)[0]
    g1, e1 = stats()
    b = checker.tonemap(hdr)[0]
    assert (a == b).all(), int((a != b).sum())
    assert g1 - g0 == w * h // 4, "the fast tone-map kernel did not run"
    share = (e1 - e0) / float(g1 - g0)
    assert 0.0 < share < 0.05, share


def test_fast_log2_error_bound(gpu):
    """Pass 2 of the two-pass fast path (k_affine_q) trusts lg2.approx to within kLg2Abs + |g| * kLg2Rel of the exact
    float(log2(double(q))).  Checked here for EVERY float q in [2^-40, 2^40] (the quotient (hdr+1e-7)/(sdr+1e-7) lives in
    [2^-31, 2^37]): the worst ratio error / bound must leave a factor 2."""
    lib = gpu.lib
    worst = C.c_float(-1.0)
    first = (127 - 40) << 23
    count = ((127 + 40) << 23) - first
    assert lib.uhdr_b200_probe_log2_fast(C.c_uint(first), C.c_uint(count), C.byref(worst)) == 0, T.gpu_err(gpu)
    assert 0.0 < worst.value <= 0.5, worst.value


def test_two_pass_takes_the_exact_log2_only_near_byte_boundaries(gpu, checker):
    """k_affine_q's screen: on noise (every gain value different) a small share of the values takes the fp64 path,
    and the map is still bit exact (the other tests); on a constant image none has to."""
    lib = gpu.lib

    def stats():
        st = (C.c_ulonglong * 2)()
        lib.uhdr_b200_generate_stats(st)
        return st[0], st[1]
    w, h = 1280, 720
    hdr, k1 = _hdr("noise", "p010", 2, A.CT_HLG, w, h)
    sdr, k2 = _sdr("noise", 0, w, h)
    v0, e0 = stats()
    g1, m1 = gpu.generate(sdr, hdr)
    v1, e1 = stats()
    g2, m2 = checker.generate(sdr, hdr)
    assert (g1 == g2).all() and T.md_equal(m1, m2)
    assert v1 - v0 == w * h * 3, "the quotient-plane path did not run"
    share = (e1 - e0) / float(v1 - v0)
    assert 0.0 < share < 0.02, share


def test_apply_8k(gpu, checker):
    """config 3 geometry: 7680x4320, RGBA8888 map at scale 1 -> RGBA half float, bit exact."""
    w, h = 7680, 4320
    sb = T.make_yuv420(w, h, "noise")
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    rs = np.random.RandomState(7)
    gm = rs.randint(0, 256, (h, w, 4)).astype(np.uint8)
    md = A.GainmapMetadata()
    for i, (mx, mn) in enumerate(((65.1, 4.9e-5), (845.9, 2.7e-3), (1283.8, 4.9e-5))):
        md.max_content_boost[i], md.min_content_boost[i], md.gamma[i] = mx, mn, 1.0
        md.offset_sdr[i] = md.offset_hdr[i] = 1e-7
    md.hdr_capacity_min, md.hdr_capacity_max, md.use_base_cg = 1.0, 4.926108, 0
    gi = T.gm_image(gm, A.CG_BT2100)
    a = gpu.apply(sdr, gi, md, A.CT_LINEAR)
    b = checker.apply(sdr, gi, md, A.CT_LINEAR)
    assert (a == b).all(), int((a != b).sum())


def test_device_log2_equals_libm(gpu, oracle_libs):
    """computeGain's `float(log2(double(q)))`: the fast gain-map kernels evaluate it with their own
    table + polynomial in fp64.  It must give the float glibc gives, on a dense sample of the
    quotient range incl. the neighbourhood of 1 and exact powers of two."""
    import ctypes as C
    o = oracle_libs.Oracle().lib
    rs = np.random.RandomState(11)
    parts = [np.exp(rs.uniform(np.log(1e-10), np.log(1e12), 6_000_000)),
             1.0 + rs.uniform(-3e-3, 3e-3, 1_000_000), 1.0 + rs.uniform(-1e-6, 1e-6, 200_000),
             2.0 ** np.arange(-30, 40), np.nextafter(np.float32(1), np.float32(0)) * np.ones(1),
             np.array([1.0, 0.69921875, 1.3984375, 0.70710678, 1.41421356])]
    x = np.ascontiguousarray(np.concatenate(parts).astype(np.float32))
    want = np.zeros_like(x)
    got = np.zeros_like(x)
    o.uo_log2_of_float(x.ctypes.data_as(C.c_void_p), want.ctypes.data_as(C.c_void_p), C.c_size_t(x.size))
    assert gpu.lib.uhdr_b200_probe_log2(x.ctypes.data_as(C.c_void_p), got.ctypes.data_as(C.c_void_p), x.size) == 0
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert bad.sum() == 0, (int(bad.sum()), x[bad][:5], got[bad][:5], want[bad][:5])


def test_apply_resized_gainmap(gpu, oracle_libs):
    """gain map whose aspect ratio differs from the base image by more than 1 %: applyGainMap first
    resizes it (resize_image, editorhelper.cpp:100-146, double-precision cubic blend).  Compared with
    the reference's own code (the C restatement does not cover this branch)."""
    ref = oracle_libs.Ref() if oracle_libs.have_ref() else None
    w, h = 256, 128
    sb = T.make_yuv420(w, h, "noise")
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    md = A.GainmapMetadata()
    for i, (mx, mn) in enumerate(((8.0, 0.5), (6.0, 0.7), (4.0, 1.0))):
        md.max_content_boost[i], md.min_content_boost[i], md.gamma[i] = mx, mn, 1.0
        md.offset_sdr[i] = md.offset_hdr[i] = 1.0 / 64
    md.hdr_capacity_min, md.hdr_capacity_max, md.use_base_cg = 1.0, 8.0, 0
    rs = np.random.RandomState(21)
    for (mw, mh, ch) in ((100, 80, 4), (64, 64, 3), (77, 13, 1), (300, 100, 4)):
        gm = rs.randint(0, 256, (mh, mw, ch)).astype(np.uint8)
        if ch == 4:
            gm[..., 3] = 255
        gi = T.gm_image(np.ascontiguousarray(gm), A.CG_BT2100)
        for ct in (A.CT_LINEAR, A.CT_PQ):
            a = gpu.apply(sdr, gi, md, ct)
            b = T.from_reference("stages/apply_resized/%dx%dx%d/ct%d" % (mw, mh, ch, ct), lambda: ref.apply(sdr, gi, md, ct))
            assert T.same(a, b), (mw, mh, ch, ct)
