"""Pins the C restatement (oracle/uhdr_oracle.c) against the reference's OWN sources compiled in
place (oracle/_ref, built by oracle/Makefile when the reference sources are present; elsewhere the
results recorded from that build, tests/golden/reference_digests.json): bit-exact LUTs, tables, gain
maps, metadata, decoded pixels, tone-mapped and re-encoded planes."""
import itertools

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A

W, H = 96, 64


@pytest.fixture(scope="module")
def pair(oracle_libs):
    """(reference build or None where it is absent, C restatement)"""
    return (oracle_libs.Ref() if oracle_libs.have_ref() else None), oracle_libs.Oracle()


def _check(key, run, R, O):
    """run(impl) -> list of results; the C restatement's list must equal the reference's"""
    got = run(O)
    want = T.from_reference("oracle_vs_ref/" + key, lambda: run(R))
    if isinstance(want, T.Recorded):
        assert T.same(got, want), key
    else:
        bad = [i for i, (a, b) in enumerate(zip(got, want)) if not T.same(a, b)]
        assert len(got) == len(want) and not bad, (key, bad[:5])


def test_luts_bitwise(pair):
    R, O = pair
    _check("luts", lambda X: [X.lut(w).view(np.uint32) for w in range(5)], R, O)


def test_idw_and_gain_lut(pair):
    import ctypes as C
    R, O = pair

    def idw(X):
        f = X.lib.ref_idw_weights if X is R else X.lib.uo_idw_weights
        out = []
        for s in (1, 2, 3, 4, 8):
            for v in range(4):
                a = np.zeros(s * s * 4, np.float32)
                f(s, v, a.ctypes.data_as(C.c_void_p))
                out.append(a.view(np.uint32))
        return out
    _check("idw_weights", idw, R, O)
    md = A.GainmapMetadata()
    for i, (mx, mn) in enumerate(((65.1, 4.9e-5), (845.9, 2.7e-3), (1283.8, 4.9e-5))):
        md.max_content_boost[i], md.min_content_boost[i], md.gamma[i] = mx, mn, 1.0

    def gain_lut(X):
        f = X.lib.ref_gain_lut if X is R else X.lib.uo_gain_lut
        f.argtypes = [C.c_void_p, C.c_float, C.c_void_p]
        out = []
        for wgt in (1.0, 0.37):
            a = np.zeros(3072, np.float32)
            f(C.byref(md), wgt, a.ctypes.data_as(C.c_void_p))
            out.append(a.view(np.uint32))
        return out
    _check("gain_lut", gain_lut, R, O)


def _inputs(kind, hct, hcg, scg, hfmt="p010"):
    if hfmt == "p010":
        hb = T.make_p010(W, H, kind)
        hdr, k = A.p010_image(hb, W, H, hcg, hct, A.CR_LIMITED)
    elif hfmt == "1010102":
        hb = T.make_rgba1010102(W, H)
        hdr, k = A.raw_image(A.FMT_RGBA1010102, hcg, hct, A.CR_FULL, W, H, [hb], [W]), hb
    else:
        hb = T.make_rgbaf16(W, H)
        hdr, k = A.raw_image(A.FMT_RGBAF16, hcg, A.CT_LINEAR, A.CR_FULL, W, H, [hb], [W]), hb
    sb = T.make_yuv420(W, H, kind)
    sdr, k2 = A.yuv420_image(sb, W, H, scg)
    return hdr, sdr, (hb, sb, k, k2)


def test_generate_matrix(pair):
    R, O = pair
    configs = list(itertools.product(["noise", "black"], [A.CT_HLG, A.CT_PQ], [0, 1, 2], [0, 1, 2], [0, 1], [1, 4], [0, 1]))

    def run(X):
        out = []
        for kind, hct, hcg, scg, multi, scale, preset in configs:
            hdr, sdr, keep = _inputs(kind, hct, hcg, scg)
            cfg = A.default_gm_config(scale_factor=scale, multichannel=multi, preset=preset)
            out.append(X.generate(sdr, hdr, cfg))
        return out
    _check("generate_matrix", run, R, O)


def test_generate_other_formats_and_options(pair):
    R, O = pair

    def run(X):
        out = []
        for hfmt, ct in (("1010102", A.CT_PQ), ("f16", A.CT_LINEAR)):
            for kw in ({}, {"multichannel": 0, "use_luminance": 0}, {"preset": 0, "gamma": 2.2}, {"gamma": 1.5},
                       {"sdr_is_601": 1, "scale_factor": 2}, {"min_content_boost": 0.5, "max_content_boost": 6.0}):
                hdr, sdr, keep = _inputs("noise", ct, 2, 0, hfmt)
                out.append(X.generate(sdr, hdr, A.default_gm_config(**kw)))
        return out
    _check("generate_other_formats", run, R, O)


def test_apply_matrix(pair):
    R, O = pair
    for multi, scale in ((1, 1), (0, 1), (1, 4), (0, 2)):
        hdr, sdr, keep = _inputs("noise", A.CT_HLG, 2, 0)
        cfg = A.default_gm_config(scale_factor=scale, multichannel=multi)
        # the reference's gain map is the input (the C restatement reproduces it: test_generate_matrix)
        g, m = T.reference_file("oracle_vs_ref/apply_input/m%d_s%d" % (multi, scale), lambda: R.generate(sdr, hdr, cfg),
                                mine=lambda: O.generate(sdr, hdr, cfg))
        maps = [g] if not multi else [g, np.concatenate([g, np.full(g.shape[:2] + (1,), 255, np.uint8)], -1)]

        def run(X):
            out = []
            for gm in maps:
                gm = np.ascontiguousarray(gm)
                for gcg, ct, boost in itertools.product([-1, 0, 2], [A.CT_LINEAR, A.CT_HLG, A.CT_PQ], [A.FLT_MAX, 2.5]):
                    gi = T.gm_image(gm, gcg)
                    out.append(X.apply(sdr, gi, m, ct, boost))
            return out
        _check("apply_matrix/m%d_s%d" % (multi, scale), run, R, O)
    # non-integer scale
    hdr, sdr, keep = _inputs("noise", A.CT_HLG, 2, 0)
    g, m = T.reference_file("oracle_vs_ref/apply_input/default", lambda: R.generate(sdr, hdr), mine=lambda: O.generate(sdr, hdr))

    def run(X):
        out = []
        for ch in (1, 3):
            crop = np.ascontiguousarray(g[:43, :64, :ch])  # keep alive: descriptors hold raw pointers
            gi = T.gm_image(crop, 2)
            out.append(X.apply(sdr, gi, m, A.CT_LINEAR))
        return out
    _check("apply_non_integer_scale", run, R, O)


def test_tonemap_and_convert(pair):
    R, O = pair

    def tonemap(X):
        out = []
        for kind, hct, hcg in itertools.product(["noise", "white"], [A.CT_HLG, A.CT_PQ], [0, 1, 2]):
            hb = T.make_p010(W, H, kind)
            hdr, k = A.p010_image(hb, W, H, hcg, hct, A.CR_LIMITED)
            out.append(X.tonemap(hdr)[0])
        hb = T.make_rgbaf16(W, H)
        hdr = A.raw_image(A.FMT_RGBAF16, 1, A.CT_LINEAR, A.CR_FULL, W, H, [hb], [W])
        out.append(X.tonemap(hdr)[0])
        return out
    _check("tonemap", tonemap, R, O)

    def convert(X):
        out = []
        for s, d in itertools.permutations([0, 1, 2], 2):
            sb = T.make_yuv420(W, H, "noise")
            out.append(X.convert_yuv(sb, W, H, s, d))
        return out
    _check("convert_yuv", convert, R, O)
