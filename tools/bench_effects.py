"""Image effects (uhdr_add_effect_*) on the device: what they cost inside uhdr_decode / uhdr_encode.

  python tools/bench_effects.py [--calls 20] [--warmup 3] [--out result.json]

Cases: 8K uhdr_decode to RGBA half-float with no effect, rotate 90, mirror, crop to 3840x2160 and resize to
3840x2160; 4K API-1 uhdr_encode with no effect and rotate 90.  Per case: the median wall time of --calls calls
after --warmup, the gather kernel's time (uhdr_b200_kernel_timing_report, one extra call with timing on), the
bytes the gathers must move (each output element read once and written once; the zero padding up to the stride
is not counted) over that time, and that rate as a fraction of a device-to-device copy of the same number of
bytes measured in the same process.  The reference build (oracle/_ref), when present, runs each case once on
the host for comparison."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import uhdr_testlib as T  # noqa: E402
from libultrahdr_b200 import ctypes_api as A  # noqa: E402

DEC_CASES = {  # 8K decode to half-float: output size of the image, of the 8K map (scale 1, RGBA8888)
    "decode_8k_none": [],
    "decode_8k_rotate90": [("rotate", 90)],
    "decode_8k_mirror": [("mirror", 1)],
    "decode_8k_crop_4k": [("crop", 1920, 1920 + 3840, 1080, 1080 + 2160)],
    "decode_8k_resize_4k": [("resize", 3840, 2160)],
}
ENC_CASES = {"encode_4k_api1_none": [], "encode_4k_api1_rotate90": [("rotate", 90)]}


def declare(lib):
    T.UhdrApi(lib)
    for f in ("uhdr_add_effect_mirror", "uhdr_add_effect_rotate", "uhdr_add_effect_crop", "uhdr_add_effect_resize"):
        getattr(lib, f).restype = A.ErrorInfo
    lib.uhdr_add_effect_crop.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]


def add(lib, h, effects):
    for e in effects:
        r = getattr(lib, "uhdr_add_effect_" + e[0])(h, *e[1:])
        assert r.error_code == 0, r.detail


def decode(lib, ci, effects):
    """-> (seconds, (w, h), (map w, h))"""
    dec = C.c_void_p(lib.uhdr_create_decoder())
    try:
        t0 = time.perf_counter()
        assert lib.uhdr_dec_set_image(dec, C.byref(ci)).error_code == 0
        add(lib, dec, effects)
        e = lib.uhdr_decode(dec)
        dt = time.perf_counter() - t0
        assert e.error_code == 0, e.detail
        d = lib.uhdr_get_decoded_image(dec).contents
        g = lib.uhdr_get_decoded_gainmap_image(dec).contents
        return dt, (d.w, d.h), (g.w, g.h, 1 if g.fmt == A.FMT_Y400 else 4)
    finally:
        lib.uhdr_release_decoder(dec)


def encode(lib, hdr, sdr, effects):
    enc = C.c_void_p(lib.uhdr_create_encoder())
    try:
        assert lib.uhdr_enc_set_raw_image(enc, C.byref(hdr), A.HDR_IMG).error_code == 0
        assert lib.uhdr_enc_set_raw_image(enc, C.byref(sdr), A.SDR_IMG).error_code == 0
        add(lib, enc, effects)
        t0 = time.perf_counter()
        e = lib.uhdr_encode(enc)
        dt = time.perf_counter() - t0
        assert e.error_code == 0, e.detail
        return dt, lib.uhdr_get_encoded_stream(enc).contents.data_sz
    finally:
        lib.uhdr_release_encoder(enc)


def copy_bandwidth(nbytes, reps=20):
    """device-to-device copy moving `nbytes` in all (nbytes/2 read + nbytes/2 written): bytes / s"""
    import torch
    n = max(1, nbytes // 2)
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        b.copy_(a)
    e.record()
    torch.cuda.synchronize()
    return 2 * n * reps / (s.elapsed_time(e) / 1e3)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def gather_ms(lib):
    r = bench.kernel_report(lib)
    n, total = r.get("effects_gather", (0, 0.0))[:2]
    return n, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-reference", action="store_true")
    args = ap.parse_args()
    assert args.calls >= 20
    gpu = T.Gpu()
    lib = gpu.lib
    declare(lib)
    ref = None if args.no_reference or not T.have_ref() else T.Ref().lib
    if ref is not None:
        declare(ref)
    res = {"gpu": gpu_info(), "calls": args.calls, "warmup": args.warmup, "cases": {}}

    def run(name, fn, gather_bytes):
        for _ in range(args.warmup):
            fn(lib)
        ts = [fn(lib)[0] for _ in range(args.calls)]
        lib.uhdr_b200_set_kernel_timing(1)
        bench.kernel_report(lib)
        fn(lib)
        launches, kms = gather_ms(lib)
        lib.uhdr_b200_set_kernel_timing(0)
        row = {"median_ms": round(statistics.median(ts) * 1e3, 3), "min_ms": round(min(ts) * 1e3, 3),
               "max_ms": round(max(ts) * 1e3, 3)}
        if gather_bytes:
            copy = copy_bandwidth(gather_bytes)
            bw = gather_bytes / (kms / 1e3)
            row.update({"gather_launches": launches, "gather_ms": round(kms, 4), "gather_bytes": gather_bytes,
                        "gather_GBps": round(bw / 1e9, 1), "copy_GBps_same_bytes": round(copy / 1e9, 1),
                        "fraction_of_copy": round(bw / copy, 3)})
        if ref is not None:
            row["reference_host_ms"] = round(fn(ref)[0] * 1e3, 1)
        res["cases"][name] = row
        print(name, json.dumps(row), flush=True)

    w, h = 7680, 4320
    p, y = bench.make_frame(w, h, 3)
    hdr, sdr, keep = bench.frame_descs(p, y, w, h)
    data = T.UhdrApi(lib).encode(hdr, sdr)
    buf = np.frombuffer(data, np.uint8).copy()
    ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
    for name, fx in DEC_CASES.items():
        _, (ow, oh), (gw, gh, gb) = decode(lib, ci, fx)
        nbytes = 2 * (ow * oh * 8 + gw * gh * gb) if fx else 0
        run(name, lambda L, fx=fx: decode(L, ci, fx), nbytes)

    w, h = 3840, 2160
    p, y = bench.make_frame(w, h, 5)
    hdr, sdr, keep = bench.frame_descs(p, y, w, h)
    for name, fx in ENC_CASES.items():
        nbytes = 2 * (w * h * 3 + w * h * 3 // 2) if fx else 0  # P010 (3 B/px) and YUV420 (1.5 B/px) intents
        run(name, lambda L, fx=fx: encode(L, hdr, sdr, fx), nbytes)

    out = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")
    print(out)


if __name__ == "__main__":
    main()
