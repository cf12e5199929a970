"""Shared helpers for the test-suite: library loading, seeded synthetic frames and thin ctypes
wrappers.  Three implementations expose the same four stage calls:

  * ``Ref``    -- oracle/_ref/libuhdr_ref_turbo.so (else libuhdr_ref.so) : the UNMODIFIED reference
                  sources compiled in place, JPEG through the real libjpeg-turbo
  * ``Oracle`` -- oracle/liboracle.so        : the plain-C restatement (the "port")
  * ``Gpu``    -- libultrahdr_b200/libuhdr_b200.so : the product (CUDA), host-buffer C ABI

so a parity test reads ``assert_same(Gpu().apply(...), Ref().apply(...))``.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from libultrahdr_b200.ctypes_api import *  # noqa: F401,F403
from libultrahdr_b200 import ctypes_api as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# two builds of the reference (oracle/Makefile): "turbo" = every reference source incl. its own
# jpeg{en,de}coderhelper.cpp on the real libjpeg-turbo (preferred); "shim" = the JPEG helper classes on
# oracle/jpeg_oracle.c (fallback when no libjpeg-turbo binary is around)
REF_SHIM_SO = os.path.join(ROOT, "oracle", "_ref", "libuhdr_ref.so")
REF_TURBO_SO = os.path.join(ROOT, "oracle", "_ref", "libuhdr_ref_turbo.so")
REF_SO = REF_TURBO_SO if os.path.exists(REF_TURBO_SO) else REF_SHIM_SO
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
GPU_SO = os.environ.get("UHDR_B200_SO") or os.path.join(ROOT, "libultrahdr_b200", "libuhdr_b200.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")
SEED = 20240607


def ensure_oracle_built():
    if not os.path.exists(ORACLE_SO):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "all"],
                              stdout=subprocess.DEVNULL)


def have_ref():
    return os.path.exists(REF_SO)


def ref_is_turbo():
    return REF_SO == REF_TURBO_SO and os.path.exists(REF_TURBO_SO)


# ------------------------------------------------------------------------------------------------
# recorded reference results (tests/golden/reference_digests.json, tests/golden/reference/)
#
# A parity test asks the reference build for its answer through from_reference() / reference_file().
# Where oracle/_ref is built, the reference computes it; everywhere else the SHA-256 recorded from an
# earlier run of the reference stands in, so the comparison is made on every machine.  Recording:
#     UHDR_RECORD_REFERENCE=<dir> python -m pytest tests      (with oracle/_ref built)
# writes <dir>/reference_digests.json and <dir>/reference/*.bin; copy them into tests/golden/.
# ------------------------------------------------------------------------------------------------
REF_DIGESTS = os.path.join(GOLDEN, "reference_digests.json")
REF_BLOBS = os.path.join(GOLDEN, "reference")
_digests_cache = None


def digest(x):
    """SHA-256 over a canonical form of bytes, arrays, strings, ctypes structures, ints and tuples of them"""
    import hashlib
    h = hashlib.sha256()

    def feed(v):
        if isinstance(v, (bytes, bytearray)):
            h.update(b"b%d:" % len(v) + bytes(v))
        elif isinstance(v, np.ndarray):
            v = np.ascontiguousarray(v)
            h.update(("a%s%s:" % (v.dtype.str, v.shape)).encode() + v.tobytes())
        elif isinstance(v, str):
            h.update(b"t%d:" % len(v) + v.encode())
        elif isinstance(v, C.Structure):
            h.update(b"s:" + bytes(v))
        elif isinstance(v, (bool, int, np.integer)):
            h.update(b"i%d;" % int(v))
        elif isinstance(v, (tuple, list)):
            h.update(b"(%d" % len(v))
            for e in v:
                feed(e)
            h.update(b")")
        elif v is None:
            h.update(b"n;")
        else:
            raise TypeError(type(v))
    feed(x)
    return h.hexdigest()


class Recorded:
    """the reference's answer known only by its recorded digest (no reference build on this machine)"""

    def __init__(self, key, sha):
        self.key, self.sha = key, sha

    def __repr__(self):
        return "Recorded(%r)" % self.key


def same(a, b):
    """a (the product's result) equals b (from_reference(), a live result or a Recorded digest)"""
    return digest(a) == (b.sha if isinstance(b, Recorded) else digest(b))


def _recorded(key):
    global _digests_cache
    if _digests_cache is None:
        import json
        _digests_cache = json.load(open(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
    sha = _digests_cache.get(key)
    assert sha is not None, "no recorded reference result for %r in %s" % (key, REF_DIGESTS)
    return sha


def _record(key, value, blob=False):
    """under UHDR_RECORD_REFERENCE=<dir>: add key -> digest (and the bytes themselves when blob) to <dir>"""
    d = os.environ.get("UHDR_RECORD_REFERENCE")
    if not d:
        return
    import json
    os.makedirs(d, exist_ok=True)
    p = os.path.join(d, "reference_digests.json")
    cur = json.load(open(p)) if os.path.exists(p) else {}
    cur[key] = digest(value)
    with open(p, "w") as f:
        json.dump(cur, f, indent=0, sort_keys=True)
        f.write("\n")
    if blob:
        os.makedirs(os.path.join(d, "reference"), exist_ok=True)
        with open(os.path.join(d, "reference", _blob_name(key)), "wb") as f:
            f.write(value)


def _blob_name(key):
    import re
    return re.sub(r"[^A-Za-z0-9_.-]+", "_", key).strip("_") + ".bin"


def from_reference(key, fn):
    """the reference's answer for `key`: fn() when the reference build is present, else its recorded digest"""
    if have_ref():
        v = fn()
        _record(key, v)
        return v
    return Recorded(key, _recorded(key))


def reference_file(key, fn, mine=None):
    """bytes (or a tuple of results) the reference produced, needed as an INPUT by a test: fn() when the
    reference build is present, and then mine() -- the product's or the C restatement's way of making
    them -- must return the same.  Otherwise mine() must reproduce the recorded digest exactly; without
    mine, the bytes stored under tests/golden/reference/ are used (and checked against the digest)."""
    if have_ref():
        v = fn()
        _record(key, v, blob=mine is None)
        if mine is not None:
            assert same(mine(), v), "%s differs from what the reference produced" % key
        return v
    sha = _recorded(key)
    if mine is not None:
        v = mine()
    else:
        with open(os.path.join(REF_BLOBS, _blob_name(key)), "rb") as f:
            v = f.read()
    assert digest(v) == sha, "%s differs from what the reference produced" % key
    return v


# ------------------------------------------------------------------------------------------------
# synthetic frames (SURVEY.md section 8d): noise / smooth / edge, seeded
# ------------------------------------------------------------------------------------------------
def make_p010(w, h, kind="noise", seed=SEED, limited=True):
    rs = np.random.RandomState(seed)
    n = w * h
    if kind == "noise":
        if limited:
            y = rs.randint(64, 941, n)
            uv = rs.randint(64, 961, n // 2)
        else:
            y = rs.randint(0, 1024, n)
            uv = rs.randint(0, 1024, n // 2)
    elif kind == "smooth":
        yy, xx = np.mgrid[0:h, 0:w]
        y = (64 + 876 * (0.5 + 0.5 * np.sin(xx / 97.0) * np.cos(yy / 61.0)) *
             (xx + yy) / (w + h)).astype(np.int64).ravel()
        cy, cx = np.mgrid[0:h // 2, 0:w // 2]
        u = 512 + 200 * np.sin(cx / 53.0)
        v = 512 + 200 * np.cos(cy / 41.0)
        uv = np.stack([u, v], -1).astype(np.int64).ravel()
    elif kind == "black":
        y = np.full(n, 64)
        uv = np.full(n // 2, 512)
    elif kind == "white":
        y = np.full(n, 940)
        uv = np.full(n // 2, 512)
    else:
        raise ValueError(kind)
    buf = np.concatenate([y, uv]).astype(np.uint16) << 6
    return np.ascontiguousarray(buf)


def make_yuv420(w, h, kind="noise", seed=SEED + 1):
    rs = np.random.RandomState(seed)
    n = w * h + 2 * (w // 2) * (h // 2)
    if kind == "noise":
        return rs.randint(0, 256, n).astype(np.uint8)
    if kind == "smooth":
        yy, xx = np.mgrid[0:h, 0:w]
        y = (255 * (0.5 + 0.5 * np.sin(xx / 97.0) * np.cos(yy / 61.0)) * (xx + yy) / (w + h))
        cy, cx = np.mgrid[0:h // 2, 0:w // 2]
        u = 128 + 50 * np.sin(cx / 53.0)
        v = 128 + 50 * np.cos(cy / 41.0)
        return np.concatenate([y.ravel(), u.ravel(), v.ravel()]).astype(np.uint8)
    if kind == "black":
        return np.concatenate([np.zeros(w * h), np.full(n - w * h, 128)]).astype(np.uint8)
    if kind == "white":
        return np.concatenate([np.full(w * h, 255), np.full(n - w * h, 128)]).astype(np.uint8)
    raise ValueError(kind)


def make_rgba1010102(w, h, seed=SEED + 2):
    rs = np.random.RandomState(seed)
    return (rs.randint(0, 1 << 30, w * h).astype(np.uint32) | np.uint32(3 << 30))


def make_rgbaf16(w, h, seed=SEED + 3):
    rs = np.random.RandomState(seed)
    px = np.ones((h * w, 4), np.float16)
    px[:, :3] = (rs.rand(h * w, 3) ** 3 * 20.0).astype(np.float16)
    # sprinkle non-finite / negative values (sanitizePixel, gainmapmath.h:588-593)
    idx = rs.randint(0, h * w, 16)
    px[idx[:4], 0] = np.inf
    px[idx[4:8], 1] = -np.inf
    px[idx[8:12], 2] = np.nan
    px[idx[12:], 0] = -1.0
    return px.view(np.uint16).reshape(-1).copy()


def make_rgba8888(w, h, seed=SEED + 4):
    rs = np.random.RandomState(seed)
    return (rs.randint(0, 1 << 24, w * h).astype(np.uint32) | np.uint32(0xFF000000))


def load_fixture_720p():
    """config 1 inputs: the reference's 1280x720 colour-bar fixtures (tests/data/raw_p010_image.p010 and
    raw_yuv420_image.yuv420 of libultrahdr), stored xz-compressed under tests/golden/."""
    import lzma
    with lzma.open(os.path.join(GOLDEN, "raw_p010_image.p010.xz")) as f:
        p = np.frombuffer(f.read(), dtype=np.uint16).copy()
    with lzma.open(os.path.join(GOLDEN, "raw_yuv420_image.yuv420.xz")) as f:
        y = np.frombuffer(f.read(), dtype=np.uint8).copy()
    return p, y


# ------------------------------------------------------------------------------------------------
class _Impl:
    """Common calling convention over a library exporting <pfx>generate_gainmap etc."""

    def __init__(self, so, pfx, mode=None):
        self.lib = C.CDLL(so) if mode is None else C.CDLL(so, mode=mode)
        self.pfx = pfx

    def f(self, name):
        return getattr(self.lib, self.pfx + name)

    def generate(self, sdr, hdr, cfg=None):
        """-> (gainmap ndarray (h,w,c) u8, GainmapMetadata)"""
        cfg = cfg or A.default_gm_config()
        s = max(1, cfg.scale_factor)
        mw, mh = sdr.w // s, sdr.h // s
        ch = 3 if cfg.multichannel else 1
        gm = np.zeros((mh, mw, ch), np.uint8)
        gmi = A.raw_image(A.FMT_RGB888 if ch == 3 else A.FMT_Y400, -1, -1, -1, mw, mh, [gm], [mw])
        md = A.GainmapMetadata()
        rc = self.f("generate_gainmap")(C.byref(sdr), C.byref(hdr), C.byref(cfg), C.byref(md),
                                        C.byref(gmi))
        assert rc == 0, f"{self.pfx}generate_gainmap rc={rc}"
        self.last_gm_desc = gmi
        return gm, md

    def apply(self, sdr, gm_img, md, out_ct, max_boost=A.FLT_MAX):
        w, h = sdr.w, sdr.h
        if out_ct == A.CT_LINEAR:
            out = np.zeros((h, w, 4), np.uint16)
            fmt = A.FMT_RGBAF16
        else:
            out = np.zeros((h, w), np.uint32)
            fmt = A.FMT_RGBA1010102
        dst = A.raw_image(fmt, -1, out_ct, A.CR_FULL, w, h, [out], [w])
        fn = self.f("apply_gainmap")
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p]
        rc = fn(C.byref(sdr), C.byref(gm_img), C.byref(md), out_ct, fmt, max_boost, C.byref(dst))
        assert rc == 0, f"{self.pfx}apply_gainmap rc={rc}"
        return out

    def tonemap(self, hdr):
        w, h = hdr.w, hdr.h
        if hdr.fmt == A.FMT_P010:
            out = np.zeros(w * h * 3 // 2, np.uint8)
            sdr, _ = A.yuv420_image(out, w, h, -1, -1, -1)
        else:
            out = np.zeros(w * h, np.uint32)
            sdr = A.raw_image(A.FMT_RGBA8888, -1, -1, -1, w, h, [out], [w])
        rc = self.f("tonemap")(C.byref(hdr), C.byref(sdr))
        assert rc == 0, f"{self.pfx}tonemap rc={rc}"
        return out, sdr

    def convert_yuv(self, buf, w, h, src_cg, dst_cg):
        b = buf.copy()
        img, _ = A.yuv420_image(b, w, h, src_cg)
        rc = self.f("convert_yuv")(C.byref(img), src_cg, dst_cg)
        assert rc == 0
        return b

    def lut(self, which):
        n = [1024, 4096, 4096, 65536, 65536][which]
        out = np.zeros(n, np.float32)
        assert self.f("lut")(which, out.ctypes.data_as(C.c_void_p), n) == 0
        return out


class Ref(_Impl):
    def __init__(self):
        super().__init__(REF_SO, "ref_")
        for n in ("srgb_oetf", "compute_gain", "hlg_ootf_1", "hlg_inv_ootf_1"):
            self.f(n).restype = C.c_float


class Oracle(_Impl):
    def __init__(self):
        super().__init__(ORACLE_SO, "uo_")
        for n in ("srgb_oetf", "compute_gain"):
            self.f(n).restype = C.c_float


class Gpu(_Impl):
    def __init__(self):
        if not os.path.exists(GPU_SO):
            raise RuntimeError("libuhdr_b200.so missing: run `python -c 'import __graft_entry__ as g;"
                               " g.build()'`")
        super().__init__(GPU_SO, "uhdr_b200_")


def gm_image(gm, cg=-1, ct=-1, rng=-1):
    """wrap a (h,w,c) u8 gain map as a raw image descriptor (c = 1, 3 or 4)."""
    h, w, c = gm.shape
    fmt = {1: A.FMT_Y400, 3: A.FMT_RGB888, 4: A.FMT_RGBA8888}[c]
    return A.raw_image(fmt, cg, ct, rng, w, h, [gm], [w])


def md_equal(a, b):
    return bytes(a) == bytes(b)


# ------------------------------------------------------------------------------------------------
# JPEG helpers: oracle codec structs (oracle/jpeg_oracle.h) and thin wrappers
# ------------------------------------------------------------------------------------------------
class JoComp(C.Structure):
    _fields_ = [(n, C.c_int) for n in "h_samp v_samp width height wblocks hblocks tq".split()]


class JoFrame(C.Structure):
    _fields_ = [(n, C.c_int) for n in "ncomp width height max_h max_v mcus_per_row mcu_rows".split()] + \
               [("comp", JoComp * 3), ("qt", (C.c_uint16 * 64) * 2)]


class JoMarker(C.Structure):
    _fields_ = [("id", C.c_uint8), ("offset", C.c_size_t), ("length", C.c_size_t)]


class JoHeader(C.Structure):
    _fields_ = [("frame", JoFrame), ("comp_id", C.c_int * 3), ("restart_interval", C.c_int),
                ("scan_offset", C.c_size_t), ("scan_end", C.c_size_t), ("markers", JoMarker * 64),
                ("nmarkers", C.c_int), ("bits", ((C.c_uint8 * 17) * 2) * 2),
                ("vals", ((C.c_uint8 * 256) * 2) * 2), ("have_tbl", (C.c_int * 2) * 2),
                ("dc_sel", C.c_int * 3), ("ac_sel", C.c_int * 3)]


def _planes3(img):
    return (C.c_void_p * 3)(img.planes[0], img.planes[1], img.planes[2]), \
        (C.c_uint * 3)(img.stride[0], img.stride[1], img.stride[2])


def oracle_forward(lib, img, quality):
    """-> (JoFrame, [coef arrays (nblocks,64) int16])"""
    f = JoFrame()
    assert lib.jo_frame_init(C.byref(f), img.fmt, img.w, img.h, quality) == 0
    coefs = [np.zeros((f.comp[c].wblocks * f.comp[c].hblocks, 64), np.int16) for c in range(f.ncomp)]
    cp = (C.c_void_p * 3)(*([c.ctypes.data for c in coefs] + [None] * (3 - f.ncomp)))
    P, S = _planes3(img)
    assert lib.jo_forward(C.byref(f), img.fmt, P, S, cp) == 0
    return f, coefs


def oracle_encode(lib, img, quality, icc=None, comment=None):
    P, S = _planes3(img)
    out = C.c_void_p()
    n = C.c_size_t()
    iccb = (C.c_uint8 * len(icc)).from_buffer_copy(icc) if icc else None
    rc = lib.jo_encode(P, S, img.w, img.h, img.fmt, quality, iccb, C.c_size_t(len(icc) if icc else 0),
                       comment, C.byref(out), C.byref(n))
    assert rc == 0
    return C.string_at(out, n.value)


def oracle_decode(lib, data):
    """-> (JoHeader, padded planes list)"""
    h = JoHeader()
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    assert lib.jo_read_header(buf, C.c_size_t(len(data)), C.byref(h)) == 0
    f = h.frame
    coefs = [np.zeros((f.comp[c].hblocks * f.comp[c].wblocks, 64), np.int16) for c in range(f.ncomp)]
    cp = (C.c_void_p * 3)(*([c.ctypes.data for c in coefs] + [None] * (3 - f.ncomp)))
    assert lib.jo_decode_coefs(buf, C.c_size_t(len(data)), C.byref(h), cp) == 0
    planes = [np.zeros((f.comp[c].hblocks * 8, f.comp[c].wblocks * 8), np.uint8) for c in range(f.ncomp)]
    pp = (C.c_void_p * 3)(*([p.ctypes.data for p in planes] + [None] * (3 - f.ncomp)))
    lib.jo_inverse(C.byref(h), cp, pp)
    return h, planes


GM_COMMENT = b"Source: google libuhdr v2.0.2, Coder: libjpeg v62, Attrib: GainMap Image"


def gpu_jpeg_forward(gpu, img, quality, frame):
    coefs = [np.zeros((frame.comp[c].wblocks * frame.comp[c].hblocks, 64), np.int16) for c in range(frame.ncomp)]
    cp = (C.c_void_p * 3)(*([c.ctypes.data for c in coefs] + [None] * (3 - frame.ncomp)))
    rc = gpu.lib.uhdr_b200_jpeg_forward(C.byref(img), quality, cp)
    assert rc == 0, gpu_err(gpu)
    return coefs


def gpu_err(gpu):
    gpu.lib.uhdr_b200_last_error.restype = C.c_char_p
    return gpu.lib.uhdr_b200_last_error()


def gpu_jpeg_encode(gpu, img, quality, icc=None):
    cap = img.w * img.h * 6 + (1 << 16)
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t()
    iccb = (C.c_uint8 * len(icc)).from_buffer_copy(icc) if icc else None
    rc = gpu.lib.uhdr_b200_jpeg_encode(C.byref(img), quality, iccb, C.c_size_t(len(icc) if icc else 0),
                                       out.ctypes.data_as(C.c_void_p), C.c_size_t(cap), C.byref(n))
    assert rc == 0, gpu_err(gpu)
    return bytes(out[:n.value])


# ------------------------------------------------------------------------------------------------
# the reference C API (ultrahdr_api.h), usable with either libuhdr_ref.so or libuhdr_b200.so
# ------------------------------------------------------------------------------------------------
class UhdrApi:
    def __init__(self, lib):
        self.lib = lib
        lib.uhdr_create_encoder.restype = C.c_void_p
        lib.uhdr_create_decoder.restype = C.c_void_p
        for f in ("uhdr_enc_set_raw_image", "uhdr_encode", "uhdr_dec_set_image", "uhdr_decode",
                  "uhdr_enc_set_quality", "uhdr_enc_set_gainmap_scale_factor", "uhdr_enc_set_preset",
                  "uhdr_enc_set_using_multi_channel_gainmap", "uhdr_dec_set_out_img_format",
                  "uhdr_dec_set_out_color_transfer", "uhdr_dec_set_out_max_display_boost", "uhdr_dec_probe",
                  "uhdr_enc_set_gainmap_gamma", "uhdr_enc_set_min_max_content_boost"):
            getattr(lib, f).restype = A.ErrorInfo
        lib.uhdr_get_encoded_stream.restype = C.POINTER(A.CompressedImage)
        lib.uhdr_get_decoded_image.restype = C.POINTER(A.RawImage)
        lib.uhdr_get_decoded_gainmap_image.restype = C.POINTER(A.RawImage)
        lib.uhdr_dec_get_gainmap_metadata.restype = C.POINTER(A.GainmapMetadata)
        lib.uhdr_enc_set_gainmap_gamma.argtypes = [C.c_void_p, C.c_float]
        lib.uhdr_dec_set_out_max_display_boost.argtypes = [C.c_void_p, C.c_float]
        lib.uhdr_enc_set_min_max_content_boost.argtypes = [C.c_void_p, C.c_float, C.c_float]

    @staticmethod
    def _ck(e):
        assert e.error_code == 0, (e.error_code, e.detail)

    def encode(self, hdr, sdr=None, quality=95, gm_quality=95, scale=1, multichannel=1, preset=None):
        L = self.lib
        enc = C.c_void_p(L.uhdr_create_encoder())
        try:
            self._ck(L.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG))
            if sdr is not None:
                self._ck(L.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG))
            self._ck(L.uhdr_enc_set_quality(enc, quality, A.BASE_IMG))
            self._ck(L.uhdr_enc_set_quality(enc, gm_quality, A.GAIN_MAP_IMG))
            self._ck(L.uhdr_enc_set_gainmap_scale_factor(enc, scale))
            self._ck(L.uhdr_enc_set_using_multi_channel_gainmap(enc, multichannel))
            if preset is not None:
                self._ck(L.uhdr_enc_set_preset(enc, preset))
            self._ck(L.uhdr_encode(enc))
            o = L.uhdr_get_encoded_stream(enc).contents
            return C.string_at(o.data, o.data_sz)
        finally:
            L.uhdr_release_encoder(enc)

    def encode_with_compressed_sdr(self, hdr, sdr_jpg, sdr=None, sdr_jpg_cg=-1, gm_quality=95, scale=1, multichannel=1):
        """encode API-2 (raw sdr intent given too) / API-3; returns the file or the error code"""
        L = self.lib
        L.uhdr_enc_set_compressed_image.restype = A.ErrorInfo
        enc = C.c_void_p(L.uhdr_create_encoder())
        try:
            self._ck(L.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG))
            if sdr is not None:
                self._ck(L.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG))
            jb = np.frombuffer(sdr_jpg, np.uint8).copy()
            ci = A.CompressedImage(jb.ctypes.data, len(sdr_jpg), len(sdr_jpg), sdr_jpg_cg, -1, -1)
            self._ck(L.uhdr_enc_set_compressed_image(enc, C.byref(ci), A.SDR_IMG))
            self._ck(L.uhdr_enc_set_quality(enc, gm_quality, A.GAIN_MAP_IMG))
            self._ck(L.uhdr_enc_set_gainmap_scale_factor(enc, scale))
            self._ck(L.uhdr_enc_set_using_multi_channel_gainmap(enc, multichannel))
            e = L.uhdr_encode(enc)
            if e.error_code:
                return int(e.error_code)
            o = L.uhdr_get_encoded_stream(enc).contents
            return C.string_at(o.data, o.data_sz)
        finally:
            L.uhdr_release_encoder(enc)

    def decode(self, data, out_fmt=A.FMT_RGBAF16, out_ct=A.CT_LINEAR, boost=None):
        L = self.lib
        dec = C.c_void_p(L.uhdr_create_decoder())
        try:
            buf = np.frombuffer(data, np.uint8).copy()
            ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
            self._ck(L.uhdr_dec_set_image(dec, C.byref(ci)))
            self._ck(L.uhdr_dec_set_out_img_format(dec, out_fmt))
            self._ck(L.uhdr_dec_set_out_color_transfer(dec, out_ct))
            if boost is not None:
                self._ck(L.uhdr_dec_set_out_max_display_boost(dec, boost))
            self._ck(L.uhdr_decode(dec))
            d = L.uhdr_get_decoded_image(dec).contents
            bpp = 8 if out_fmt == A.FMT_RGBAF16 else 4
            px = np.ctypeslib.as_array(C.cast(d.planes[0], C.POINTER(C.c_uint8)), (d.h, d.stride[0] * bpp)).copy()
            g = L.uhdr_get_decoded_gainmap_image(dec).contents
            gb = 1 if g.fmt == A.FMT_Y400 else 4
            gm = np.ctypeslib.as_array(C.cast(g.planes[0], C.POINTER(C.c_uint8)), (g.h, g.stride[0] * gb)).copy()
            md = A.GainmapMetadata.from_buffer_copy(bytes(L.uhdr_dec_get_gainmap_metadata(dec).contents))
            return px[:, :d.w * bpp], gm[:, :g.w * gb], md, d.cg
        finally:
            L.uhdr_release_decoder(dec)
