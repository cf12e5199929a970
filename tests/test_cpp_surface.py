"""The reference's C++ surface (ultrahdr::JpegR incl. the deprecated jr_* overloads, UltraHdr stage
members, JpegEncoderHelper) exported by libuhdr_b200.so: tests/cpp/jpegr_surface_test.cpp -- one source
file that compiles unmodified against the reference's headers AND against include/ -- must print, built
against include/ + libuhdr_b200.so, the lines it printed when built against the reference
(tests/golden/jpegr_surface_ref.txt, made by tools/make_surface_golden.py)."""
import os
import shutil
import subprocess

import pytest

import uhdr_testlib as T

SRC = os.path.join(T.ROOT, "tests", "cpp", "jpegr_surface_test.cpp")
GOLD = os.path.join(T.ROOT, "tests", "golden", "jpegr_surface_ref.txt")


def _build(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    import __graft_entry__ as g
    g.build()
    exe = str(tmp_path / "jpegr_surface_test")
    libdir = os.path.join(T.ROOT, "libultrahdr_b200")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(T.ROOT, "include"), SRC, os.path.join(libdir, "libuhdr_b200.so"),
           "-Wl,-rpath," + libdir, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_surface_compiles_and_links_against_include(tmp_path):
    """no GPU needed: every class, overload and constant the reference's integration test uses is declared
    by include/ultrahdr/*.h and exported by the shared library"""
    exe = _build(tmp_path)
    out = subprocess.run(["nm", "-D", "--defined-only", "-C", os.path.join(T.ROOT, "libultrahdr_b200", "libuhdr_b200.so")],
                         capture_output=True, text=True).stdout
    for sym in ("ultrahdr::JpegR::JpegR(", "ultrahdr::JpegR::encodeJPEGR(", "ultrahdr::JpegR::decodeJPEGR(", "ultrahdr::JpegR::getJPEGRInfo(",
                "ultrahdr::UltraHdr::generateGainMap(", "ultrahdr::UltraHdr::applyGainMap(", "ultrahdr::UltraHdr::toneMap(",
                "ultrahdr::UltraHdr::convertYuv(", "ultrahdr::UltraHdr::parseGainMapMetadata(", "ultrahdr::JpegEncoderHelper::compressImage(",
                "ultrahdr::JpegDecoderHelper::decompressImage(", "ultrahdr::globalTonemap("):
        assert sym in out, sym
    assert out.count("ultrahdr::JpegR::encodeJPEGR(") == 10  # five current + five deprecated overloads
    assert os.path.exists(exe)


@pytest.mark.gpu
def test_surface_behaves_like_the_reference(gpu, tmp_path):
    # the reference's 1280x720 fixtures (stored compressed in tests/golden), as the files the program reads
    pb, yb = T.load_fixture_720p()
    p, y = str(tmp_path / "raw_p010_image.p010"), str(tmp_path / "raw_yuv420_image.yuv420")
    pb.tofile(p)
    yb.tofile(y)
    exe = _build(tmp_path)
    r = subprocess.run([exe, p, y], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    got = r.stdout.strip().splitlines()
    want = open(GOLD).read().strip().splitlines()
    assert got == want, [(a, b) for a, b in zip(got, want) if a != b][:5]
