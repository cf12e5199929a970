"""Host-side half of the decoder (container split, marker parsing, ISO 21496-1 metadata codec, EXIF /
ICC extraction) needs no GPU: uhdr_dec_probe of libuhdr_b200.so against the reference's uhdr_dec_probe
on files written by the reference encoder."""
import ctypes as C

import numpy as np
import pytest

import uhdr_testlib as T
from libultrahdr_b200 import ctypes_api as A


def _probe(lib, data):
    lib.uhdr_create_decoder.restype = C.c_void_p
    for f in ("uhdr_dec_set_image", "uhdr_dec_probe"):
        getattr(lib, f).restype = A.ErrorInfo
    for f in ("uhdr_dec_get_exif", "uhdr_dec_get_icc", "uhdr_dec_get_base_image", "uhdr_dec_get_gainmap_image"):
        getattr(lib, f).restype = C.POINTER(A.MemBlock)
    lib.uhdr_dec_get_gainmap_metadata.restype = C.POINTER(A.GainmapMetadata)
    dec = C.c_void_p(lib.uhdr_create_decoder())
    try:
        buf = np.frombuffer(data, np.uint8).copy()
        ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
        e = lib.uhdr_dec_set_image(dec, C.byref(ci))
        assert e.error_code == 0, e.detail
        e = lib.uhdr_dec_probe(dec)
        if e.error_code != 0:
            return {"error": e.error_code}
        out = {"dims": (lib.uhdr_dec_get_image_width(dec), lib.uhdr_dec_get_image_height(dec),
                        lib.uhdr_dec_get_gainmap_width(dec), lib.uhdr_dec_get_gainmap_height(dec))}
        for name in ("exif", "icc", "base_image", "gainmap_image"):
            blk = getattr(lib, "uhdr_dec_get_" + name)(dec)
            out[name] = C.string_at(blk.contents.data, blk.contents.data_sz) if blk and blk.contents.data_sz else b""
        md = lib.uhdr_dec_get_gainmap_metadata(dec)
        out["md"] = A.GainmapMetadata.from_buffer_copy(bytes(md.contents)) if md else None
        return out
    finally:
        lib.uhdr_release_decoder(dec)


def _summary(p):
    """what a caller of uhdr_dec_probe gets: the verdict, or dimensions, metadata and the four blocks"""
    if "error" in p:
        return ("error", p["error"])
    return (p["dims"], p["md"], p["exif"], p["icc"], p["base_image"], p["gainmap_image"])


def _ref_lib(oracle_libs):
    """the reference build, or None where it is absent (recorded results stand in)"""
    return oracle_libs.Ref().lib if oracle_libs.have_ref() else None


def _seed_file(oracle_libs, w=64, h=64):
    """a JPEG/R the reference encoder wrote from the smooth test frames"""
    hb = T.make_p010(w, h, "smooth")
    sb = T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    return T.reference_file("probe/file_%dx%d" % (w, h), lambda: T.UhdrApi(oracle_libs.Ref().lib).encode(hdr, sdr))


@pytest.mark.parametrize("opts", [{}, {"scale": 4, "multichannel": 0}, {"preset": A.USAGE_REALTIME, "quality": 60}, {"api0": True}])
def test_probe_matches_reference(oracle_libs, opts):
    import os
    ref_lib = _ref_lib(oracle_libs)
    mine_lib = C.CDLL(os.path.join(oracle_libs.ROOT, "libultrahdr_b200", "libuhdr_b200.so"))
    w, h = 320, 192
    hb = T.make_p010(w, h, "smooth")
    sb = T.make_yuv420(w, h, "smooth")
    hdr, k1 = A.p010_image(hb, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(sb, w, h, A.CG_BT709)
    o = dict(opts)
    api0 = o.pop("api0", False)
    key = "probe/match/%s" % sorted(opts.items())
    data = T.reference_file(key + "/file", lambda: T.UhdrApi(ref_lib).encode(hdr, None if api0 else sdr, **o))
    a = _probe(mine_lib, data)
    assert "error" not in a, a
    b = T.from_reference(key + "/probe", lambda: _summary(_probe(ref_lib, data)))
    assert T.same(_summary(a), b)


def test_probe_rejects_what_the_reference_rejects(oracle_libs):
    import os
    ref_lib = _ref_lib(oracle_libs)
    mine_lib = C.CDLL(os.path.join(oracle_libs.ROOT, "libultrahdr_b200", "libuhdr_b200.so"))
    good = _seed_file(oracle_libs)
    second = good.index(b"\xff\xd8", 4)
    # inputs the reference build itself handles: compare the verdicts
    for name, bad in (("primary_only", good[:second]),   # primary image only: no gain map
                      ("zeros", b"\x00" * 64)):           # not a JPEG at all
        a = _probe(mine_lib, bad)
        b = T.from_reference("probe/verdict/" + name, lambda: "error" in _probe(ref_lib, bad))
        assert T.same("error" in a, b), (name, a.get("error"), b)
    # truncated streams (the reference build used as checker crashes on these): must be refused cleanly
    for bad in (good[:200], good[:second] + good[second:second + 40], good[:3], good[:second + 2]):
        assert "error" in _probe(mine_lib, bad), len(bad)


def test_probe_survives_mutated_streams(oracle_libs):
    """byte flips, truncations and deletions all over a valid file: the host-side parsers (container
    split, marker walk, ISO 21496-1 metadata, ICC gamut) must answer with a verdict, never crash."""
    import os
    mine_lib = C.CDLL(os.path.join(oracle_libs.ROOT, "libultrahdr_b200", "libuhdr_b200.so"))
    good = bytearray(_seed_file(oracle_libs))
    n = len(good)
    rs = np.random.RandomState(20240607)
    verdicts = [0, 0]
    for it in range(600):
        bad = bytearray(good)
        mode = it % 4
        if mode == 0:
            for _ in range(rs.randint(1, 6)):
                bad[rs.randint(0, n)] = rs.randint(0, 256)
        elif mode == 1:
            bad = bad[:rs.randint(1, n)]
        elif mode == 2:
            a = rs.randint(0, n)
            del bad[a:min(n, a + rs.randint(1, 64))]
        else:
            a = rs.randint(0, min(n, 1200))   # marker / metadata region
            for _ in range(rs.randint(1, 4)):
                bad[min(len(bad) - 1, a + rs.randint(0, 32))] = rs.randint(0, 256)
        if not bad:
            continue
        verdicts["error" in _probe(mine_lib, bytes(bad))] += 1
    assert verdicts[0] > 0 and verdicts[1] > 0, verdicts


def test_host_parsers_under_sanitizers(oracle_libs, tmp_path):
    """the same mutations, 6000 of them, through the host sources compiled with AddressSanitizer and
    UndefinedBehaviorSanitizer (tests/cpp/host_parsers_fuzz.cpp): no report may appear."""
    import os
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    root = oracle_libs.ROOT
    seed = tmp_path / "seed.jpg"
    seed.write_bytes(_seed_file(oracle_libs))
    exe = str(tmp_path / "fuzz")
    csrc = os.path.join(root, "libultrahdr_b200", "csrc")
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-I", csrc,
           "-I", os.path.join(root, "include"), "-I", "/usr/local/cuda/include",
           os.path.join(root, "tests", "cpp", "host_parsers_fuzz.cpp"), os.path.join(csrc, "container.cpp"),
           os.path.join(csrc, "jpeg_host.cpp"), "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0 and "sanitize" in r.stderr:
        pytest.skip("toolchain without sanitizer runtimes")
    assert r.returncode == 0, r.stderr[-2000:]
    r = subprocess.run([exe, str(seed), "7", "6000"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "harness done" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])
    assert "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-2000:]
    # the heap-free writers (fixed-capacity sinks) at every capacity, and a header with more APPn markers than the list keeps
    r = subprocess.run([exe, str(seed), "writers"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "writers rc=0" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])
    assert "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-2000:]
    # regression (round-1 advisor finding): a DHT table that no scan component selects may be malformed
    # (libjpeg derives tables lazily, so such a file is legal); the table builders must never see it.
    # Gray JPEG using tables DC0/AC0 + an extra DC table id 1 whose 255 one-bit codes describe no prefix code.
    olib = oracle_libs.Oracle().lib
    g = (np.add.outer(np.arange(32), np.arange(32)) * 3 % 256).astype(np.uint8)
    img = A.raw_image(A.FMT_Y400, -1, -1, 1, 32, 32, [g], [32])
    good = T.oracle_encode(olib, img, 90)
    sos = good.index(b"\xff\xda")
    bogus = b"\xff\xc4" + (2 + 17 + 255).to_bytes(2, "big") + bytes([0x01, 255] + [0] * 15) + bytes(range(255))
    for name, table in (("unused", bogus), ("unused_ac", bogus.replace(b"\x01\xff", b"\x11\xff", 1))):
        poc = tmp_path / ("poc_%s.jpg" % name)
        poc.write_bytes(good[:sos] + table + good[sos:])
        r = subprocess.run([exe, str(poc), "single"], capture_output=True, text=True, timeout=60)
        assert r.returncode == 0 and "single rc=0" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])
        assert "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-2000:]
