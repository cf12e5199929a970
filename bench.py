#!/usr/bin/env python
"""bench.py -- headline benchmark of libuhdr_b200 (contract: see the task statement).

Workload (BASELINE.json metric "MPix/s encode(API-1)+decode at 4K/8K"): one *step* = API-1 encode of
a batch of F independent 3840x2160 frames (P010 HLG BT.2100 limited range + YUV420 BT.709, default
encoder settings: q95/q95, multichannel gain map at scale 1, BEST_QUALITY two-pass) per GPU, through
the drop-in C ABI (uhdr_create_encoder / uhdr_enc_set_raw_image / uhdr_encode /
uhdr_get_encoded_stream).  Frames shard across ranks with no data-path collective ("scaling":
"weak"); the only collective is one NCCL broadcast of the OETF/inverse-OETF LUT blob at start-up.

  value : MPix/s with inputs already resident in HBM (uploaded by uhdr_enc_set_raw_image outside the
          timed region; the timed region is uhdr_encode ... uhdr_get_encoded_stream: kernels,
          entropy coding, D2H of the streams, container assembly).
  e2e   : the same metric through the whole C-ABI sequence with HOST buffers every step (H2D of both
          inputs and D2H of the stream inside the timed region).
  extra : 8K decode (config 3) and 4K API-0 (config 2) device-resident numbers + applyGainMap roofline.

`--impl reference` times the reference's own CPU implementation (oracle/_ref: the reference sources
compiled in place, its JPEG helper classes on the real libjpeg-turbo binary of this image) on all host
threads.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from libultrahdr_b200 import ctypes_api as A  # noqa: E402

W4K, H4K = 3840, 2160
W8K, H8K = 7680, 4320
MPIX_4K = W4K * H4K / 1e6


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------------------------------------
# synthetic frames: natural-image-like (smooth + texture) so the entropy coder sees realistic
# statistics; every frame differs (phase shift) so a batch does not fit in L2 (8 x 37 MB > 126 MB)
# ------------------------------------------------------------------------------------------------
def make_frame(w, h, idx):
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    ph = 0.37 * idx
    base = 0.5 + 0.35 * np.sin(xx / 211.0 + ph) * np.cos(yy / 173.0 - ph) + 0.1 * np.sin((xx + yy) / 37.0 + ph)
    rs = np.random.RandomState(1000 + idx)
    tex = rs.randn(h // 8, w // 8).astype(np.float32)
    tex = np.kron(tex, np.ones((8, 8), np.float32)) * 0.02 + rs.randn(h, w).astype(np.float32) * 0.004
    lum = np.clip(base + tex, 0, 1)
    y10 = (64 + 876 * lum).astype(np.uint16)
    cy, cx = np.mgrid[0:h // 2, 0:w // 2].astype(np.float32)
    u = 512 + 180 * np.sin(cx / 97.0 + ph)
    v = 512 + 180 * np.cos(cy / 83.0 - ph)
    uv10 = np.stack([u, v], -1).astype(np.uint16)
    p010 = np.concatenate([y10.ravel(), uv10.ravel()]).astype(np.uint16) << 6
    # sdr: a tone-compressed rendition of the same scene
    sl = np.clip(lum ** 0.8 * 0.9, 0, 1)
    y8 = (255 * sl).astype(np.uint8)
    u8 = (128 + 45 * np.sin(cx / 97.0 + ph)).astype(np.uint8)
    v8 = (128 + 45 * np.cos(cy / 83.0 - ph)).astype(np.uint8)
    yuv = np.concatenate([y8.ravel(), u8.ravel(), v8.ravel()])
    return np.ascontiguousarray(p010), np.ascontiguousarray(yuv)


def frame_descs(p010, yuv, w, h):
    hdr, k1 = A.p010_image(p010, w, h, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
    sdr, k2 = A.yuv420_image(yuv, w, h, A.CG_BT709)
    return hdr, sdr, (k1, k2)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region: NVML every 10 ms (what nvidia-smi's
    clocks.sm / clocks_event_reasons.* print), falling back to nvidia-smi itself."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index, nvml_handle=None):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.h = nvml_handle
        self.samples = []   # (sm_mhz, max_mhz, [reason flags])
        self.stop_flag = False

    def _nvml(self):
        import pynvml as N
        sm = N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM)
        mx = N.nvmlDeviceGetMaxClockInfo(self.h, N.NVML_CLOCK_SM)
        r = N.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        flags = [bool(r & N.nvmlClocksThrottleReasonHwSlowdown), bool(r & N.nvmlClocksThrottleReasonHwThermalSlowdown),
                 bool(r & N.nvmlClocksThrottleReasonSwThermalSlowdown), bool(r & N.nvmlClocksThrottleReasonSwPowerCap)]
        self.samples.append((int(sm), int(mx), flags))

    def _smi(self):
        o = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in o.strip().split(",")]
        if len(f) >= 6 and f[0].isdigit() and f[1].isdigit():
            self.samples.append((int(f[0]), int(f[1]), [x.lower().startswith("active") for x in f[2:6]]))

    def run(self):
        while not self.stop_flag:
            try:
                if self.h is not None:
                    self._nvml()
                    time.sleep(0.01)
                    continue
                self._smi()
            except Exception:  # noqa: BLE001
                if self.h is not None:
                    self.h = None   # NVML query failed: use nvidia-smi from here on
                    continue
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[2][i] for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": max(s[1] for s in self.samples),
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.h is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
def load_api(path):
    lib = C.CDLL(path)
    import uhdr_testlib as T
    return T.UhdrApi(lib), lib


def run_threads(n, fn, before_start=None):
    """n host threads run fn(i).  With before_start: the threads are created first and wait at a gate; before_start()
    runs (synchronise the device / the ranks, read the clock), then the gate opens -- thread creation stays outside
    the timed region, the work does not."""
    errs = []
    gate = threading.Barrier(n + 1) if before_start else None

    def wrap(i):
        try:
            if gate:
                gate.wait()
            fn(i)
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))
    th = [threading.Thread(target=wrap, args=(i,)) for i in range(n)]
    for t in th:
        t.start()
    if gate:
        before_start()
        gate.wait()
    for t in th:
        t.join()
    if errs:
        raise RuntimeError(errs[0])


class EncoderSlot:
    """one reusable encoder handle of the C API"""

    def __init__(self, lib):
        self.lib = lib
        self.h = C.c_void_p(lib.uhdr_create_encoder())

    def set_inputs(self, hdr, sdr):
        L = self.lib
        e = L.uhdr_enc_set_raw_image(self.h, C.byref(hdr), A.HDR_IMG)
        assert e.error_code == 0, e.detail
        if sdr is not None:
            e = L.uhdr_enc_set_raw_image(self.h, C.byref(sdr), A.SDR_IMG)
            assert e.error_code == 0, e.detail

    def encode(self):
        e = self.lib.uhdr_encode(self.h)
        assert e.error_code == 0, e.detail
        return self.lib.uhdr_get_encoded_stream(self.h).contents.data_sz

    def rearm(self):
        assert self.lib.uhdr_b200_enc_rearm(self.h) == 0

    def reset(self):
        self.lib.uhdr_reset_encoder(self.h)


def kernel_report(lib, reset=True):
    buf = C.create_string_buffer(1 << 16)
    n = lib.uhdr_b200_kernel_timing_report(buf, C.c_size_t(len(buf)), 1 if reset else 0)
    out = {}
    if n > 0:
        for line in buf.value.decode().strip().split("\n"):
            f = line.split()   # name count total_ms [min_ms max_ms]
            out[f[0]] = (int(f[1]), float(f[2])) + tuple(float(x) for x in f[3:5])
    return out


# algorithmic (compulsory) bytes per launch, per full-resolution pixel of a 4K API-1 frame with the
# default settings (P010 + YUV420 in, RGB888 gain map at scale 1); derivations in DESIGN.md section 3
ALG_BYTES_PER_PX = {
    "gainmap_pass1": 4.5 + 12.0,        # read P010 3 + YUV420 1.5, write 3 float gains
    "gainmap_affine": 12.0 + 3.0,       # read gains, write RGB888
    "gainmap_onepass": 4.5 + 3.0,
    "yuv_convert": 3.0,                 # in place: 1.5 read + 1.5 written
    "tonemap": 4.5,
    "apply_gainmap": 13.5,              # YUV420 1.5 + RGBA8888 map 4 read, RGBA-F16 8 written
    # SURVEY 8(d): FDCT+quant = 1 B/sample in + 2 B/sample out (4.5 B/px for 4:2:0, 9 B/px for 3-comp 4:4:4), avg of
    # the two launches.  The kernel is fused with the entropy coder's front end and writes 16 B per block instead
    # of 128 B of coefficients, so its real DRAM traffic (roofline.traffic, ncu) is far below this figure.
    "fdct_quant": (4.5 + 9.0) / 2,
    # entropy coding proper: 16 B of block meta in (0.25 B/sample: 0.375 / 0.75 B/px) + the stream out (~0.28 B/px)
    "huff_encode": (0.375 + 0.75) / 2 + 0.28,
}
DATA_KERNELS = ("gainmap_pass1", "gainmap_affine", "fdct_quant", "huff_encode", "yuv_convert")


def load_traffic():
    """dram__bytes_read+write per launch from the committed ncu capture (profiles/), if any"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:  # noqa: BLE001
        return {}


def nvml_handle(torch, local):
    """NVML handle of torch's device `local` (matched by PCI address, so CUDA_VISIBLE_DEVICES is honoured)"""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            pr = torch.cuda.get_device_properties(local)
            bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            try:
                return pynvml.nvmlDeviceGetHandleByPciBusId(bus)
            except TypeError:
                return pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:  # noqa: BLE001
            return pynvml.nvmlDeviceGetHandleByIndex(local)
    except Exception:  # noqa: BLE001
        return None


def bind_to_gpu_numa_node(h, local):
    """one process per GPU: run on (and first-touch pinned memory from) the CPU cores NVML names as
    closest to that GPU.  Returns a short description for the config, or the reason it was skipped."""
    try:
        import pynvml
        if h is None:
            return "unchanged (no NVML handle)"
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus:
            return "unchanged (empty NVML cpu set)"
        os.sched_setaffinity(0, cpus)
        return "%d cpus near gpu %d (%d-%d)" % (len(cpus), local, cpus[0], cpus[-1])
    except Exception as e:  # noqa: BLE001
        return "unchanged (%s)" % type(e).__name__


def bench_b200(args, rank, world):
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
    import torch
    import torch.distributed as dist
    import __graft_entry__ as G
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    nvh = nvml_handle(torch, local)
    affinity = bind_to_gpu_numa_node(nvh, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        every = [None] * world
        dist.all_gather_object(every, affinity)
        affinity = every   # one entry per rank
    so = os.path.join(ROOT, "libultrahdr_b200", "libuhdr_b200.so")
    if not os.path.exists(so):
        G.build()
    api, lib = load_api(so)
    lib.uhdr_b200_kernel_launches.restype = C.c_ulonglong
    lib.uhdr_b200_lut_blob_floats.restype = C.c_size_t

    # --- the one collective: rank 0 builds the LUT blob with the reference's host expressions,
    #     broadcasts it over NCCL, every rank installs the received copy ---
    nlut = lib.uhdr_b200_lut_blob_floats()
    lut = torch.empty(nlut, dtype=torch.float32, device="cuda")
    if rank == 0:
        host = np.zeros(nlut, np.float32)
        assert lib.uhdr_b200_build_lut_blob(host.ctypes.data_as(C.c_void_p)) == 0
        lut.copy_(torch.from_numpy(host))
    if world > 1:
        dist.broadcast(lut, src=0)
    torch.cuda.synchronize()
    assert lib.uhdr_b200_install_lut_blob_dev(C.c_void_p(lut.data_ptr())) == 0

    F = args.frames
    slots_n = min(args.slots, F)

    def pinned(a):
        # the end-to-end arm copies from PINNED host memory (contract: "host->device copy of that
        # step's inputs from pinned host memory")
        t = torch.from_numpy(a).pin_memory()
        return t.numpy(), t
    frames, _pins = [], []
    for i in range(F):
        p, y = make_frame(W4K, H4K, rank * F + i)
        (p, tp), (y, ty) = pinned(p), pinned(y)
        frames.append((p, y))
        _pins.append((tp, ty))
    descs = [frame_descs(p, y, W4K, H4K) for (p, y) in frames]
    in_bytes = sum(p.nbytes + y.nbytes for (p, y) in frames)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(t):
        if world == 1:
            return t
        x = torch.tensor([t], dtype=torch.float64, device="cuda")
        dist.all_reduce(x, op=dist.ReduceOp.MAX)
        return float(x.item())

    # ---------------- device-resident: one handle per frame, inputs uploaded once ----------------
    handles = [EncoderSlot(lib) for _ in range(F)]
    for hnd, (hdr, sdr, _) in zip(handles, descs):
        hnd.set_inputs(hdr, sdr)
    out_bytes = [0] * F

    # K steps = K passes over the rank's F frames.  The host threads (one per encoder slot) are started once per
    # timed region and walk their share of every step back to back: a thread join after every step would idle the
    # device for one encode latency per step, which is an artefact of the harness, not of the library.
    def resident_steps(k, before_start=None):
        def work(s):
            for _ in range(k):
                for i in range(s, F, slots_n):
                    handles[i].rearm()
                    out_bytes[i] = handles[i].encode()
        run_threads(slots_n, work, before_start)

    resident_steps(args.warmup)
    lib.uhdr_b200_set_kernel_timing(0)
    sampler = ClockSampler(local, nvh)
    sampler.start()
    clock = {}

    def open_timed_region():
        barrier()
        clock["l0"] = lib.uhdr_b200_kernel_launches()
        clock["t0"] = time.perf_counter()
    resident_steps(args.steps, open_timed_region)
    torch.cuda.synchronize()
    t_res = max_over_ranks(time.perf_counter() - clock["t0"])
    # what the last timed step handed its callers: one JPEG/R stream per frame
    # (rank 0's frames only: the dump stays within its size budget whatever the number of ranks)
    last_streams = [stream_bytes(lib, hnd.h) for hnd in handles] if args.dump_outputs and rank == 0 else None
    l0 = clock["l0"]
    launches = lib.uhdr_b200_kernel_launches() - l0
    lib.uhdr_b200_set_kernel_timing(1)
    barrier()
    sampler.stop_flag = True
    kt_busy = kernel_report(lib)
    # kernel durations for the roofline: the same frames, ONE encoder in flight, so that the CUDA
    # events around each launch are not stretched by kernels of other streams sharing the SMs
    for _ in range(2):
        for i in range(F):
            handles[i].rearm()
            handles[i].encode()
    kernel_report(lib)
    for _ in range(args.steps):
        for i in range(F):
            handles[i].rearm()
            handles[i].encode()
    kt = kernel_report(lib)
    lib.uhdr_b200_set_kernel_timing(0)
    value = world * F * args.steps * MPIX_4K / t_res

    # ---------------- end to end: host buffers through the whole C-ABI sequence -----------------
    e2e_slots = [EncoderSlot(lib) for _ in range(slots_n)]
    e2e_out = [0] * F

    def e2e_steps(k, before_start=None):
        def work(s):
            sl = e2e_slots[s]
            for _ in range(k):
                for i in range(s, F, slots_n):
                    sl.reset()
                    sl.set_inputs(descs[i][0], descs[i][1])
                    e2e_out[i] = sl.encode()
        run_threads(slots_n, work, before_start)

    e2e_steps(max(1, args.warmup // 2))

    def open_e2e_region():
        barrier()
        clock["t0"] = time.perf_counter()
    e2e_steps(args.steps, open_e2e_region)
    torch.cuda.synchronize()
    t_e2e = max_over_ranks(time.perf_counter() - clock["t0"])
    e2e_value = world * F * args.steps * MPIX_4K / t_e2e

    # ---------------- decode arm of the metric (config 3): 8K JPEG/R -> RGBA half float ------------
    # through uhdr_dec_set_image / uhdr_decode / uhdr_get_decoded_image with the compressed stream in
    # host memory and the pixels delivered to host memory (D2H of 265 MB per image inside the timed
    # region); 4 reused decoder handles (host threads) per GPU, every rank decodes its own images
    dec_handles, dec_per = 4, max(2, min(6, args.steps))
    p8, y8 = make_frame(W8K, H8K, 7 + rank)
    h8, s8, _k8 = frame_descs(p8, y8, W8K, H8K)
    data8 = api.encode(h8, s8)
    del p8, y8, h8, s8, _k8
    buf8 = np.frombuffer(data8, np.uint8).copy()
    ci8 = A.CompressedImage(buf8.ctypes.data, len(data8), len(data8), -1, -1, -1)
    decs = [C.c_void_p(lib.uhdr_create_decoder()) for _ in range(dec_handles)]

    def dec_round(n):
        def work(i):
            for _ in range(n):
                lib.uhdr_reset_decoder(decs[i])
                assert lib.uhdr_dec_set_image(decs[i], C.byref(ci8)).error_code == 0
                e = lib.uhdr_decode(decs[i])
                assert e.error_code == 0, e.detail
                assert lib.uhdr_get_decoded_image(decs[i]).contents.w == W8K
        run_threads(dec_handles, work)
    dec_round(2)
    barrier()
    t0 = time.perf_counter()
    dec_round(dec_per)
    torch.cuda.synchronize()
    t_dec = max_over_ranks(time.perf_counter() - t0)
    dec_value = world * dec_handles * dec_per * (W8K * H8K / 1e6) / t_dec
    if last_streams is not None:
        dump_outputs(args.dump_outputs, last_streams, lib.uhdr_get_decoded_image(decs[0]).contents)
        del last_streams
    for d in decs:
        lib.uhdr_release_decoder(d)

    # what the link itself gives on this box: plain pinned<->device copies of 256 MB, CUDA events
    def pcie_probe():
        """pinned<->device copies of 256 MB, CUDA events: one stream, and four streams with 64 MB each (several DMA
        queues in flight, like the encoder slots); best of 3 trials of 4 copies each -- single trials on these
        boxes scatter between 33 and 56 GB/s"""
        try:
            n, parts = 256 << 20, 4
            hbuf = torch.empty(n, dtype=torch.uint8).pin_memory()
            dbuf = torch.empty(n, dtype=torch.uint8, device="cuda")
            streams = [torch.cuda.Stream() for _ in range(parts)]
            res = {}
            for name, (dst, src) in (("h2d_gbs", (dbuf, hbuf)), ("d2h_gbs", (hbuf, dbuf))):
                for multi in (False, True):
                    best = 0.0
                    for trial in range(4):
                        torch.cuda.synchronize()
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        if multi:
                            for st in streams:
                                st.wait_event(a)
                            for _ in range(4):
                                for k, st in enumerate(streams):
                                    with torch.cuda.stream(st):
                                        lo, hi = k * (n // parts), (k + 1) * (n // parts)
                                        dst[lo:hi].copy_(src[lo:hi], non_blocking=True)
                            for st in streams:
                                torch.cuda.current_stream().wait_stream(st)
                        else:
                            for _ in range(4):
                                dst.copy_(src, non_blocking=True)
                        b.record()
                        torch.cuda.synchronize()
                        if trial:   # first trial warms up
                            best = max(best, 4 * n / (a.elapsed_time(b) * 1e-3) / 1e9)
                    res[name + ("_4streams" if multi else "")] = round(best, 1)
            res["h2d_gbs"] = max(res["h2d_gbs"], res.pop("h2d_gbs_4streams"))
            res["d2h_gbs"] = max(res["d2h_gbs"], res.pop("d2h_gbs_4streams"))
            res["how"] = "best of one-stream and four-stream pinned copies of 256 MB, best of 3 trials"
            return res
        except Exception as e:  # noqa: BLE001
            return {"error": repr(e)}
    # every rank probes its own link AT THE SAME TIME (barrier first), so that the N-GPU end-to-end number can
    # be read against what the host (sockets' DRAM, PCIe root complexes) gives N GPUs together
    barrier()
    pcie = pcie_probe()
    if world > 1:
        every = [None] * world
        dist.all_gather_object(every, pcie)
        pcie = {"concurrent_per_rank": every,
                "h2d_gbs_sum": round(sum(e.get("h2d_gbs", 0.0) for e in every), 1),
                "d2h_gbs_sum": round(sum(e.get("d2h_gbs", 0.0) for e in every), 1)}
        barrier()
        solo = pcie_probe() if rank == 0 else None     # rank 0 alone, the other ranks idle at the next barrier
        barrier()
        pcie["rank0_alone"] = solo

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    hbm = pk["hbm_gbs"]
    traffic = load_traffic()
    kernels = {}
    for k, v in sorted(kt.items()):
        cnt, ms = v[:2]
        avg_ms = ms / cnt
        e = {"launches_per_frame": round(cnt / (F * args.steps), 2), "avg_ms": round(avg_ms, 4)}
        bpp = ALG_BYTES_PER_PX.get(k)
        if bpp:
            ach = bpp * W4K * H4K / (avg_ms * 1e-3) / 1e9
            e.update({"alg_bytes_per_launch": int(bpp * W4K * H4K), "achieved_gbs": round(ach, 1), "frac_of_hbm": round(ach / hbm, 4)})
        kernels[k] = e
    # dominant kernel = largest share of the single-stream step among the data-moving kernels
    cand = [(kt[k][1], k) for k in DATA_KERNELS if k in kt]
    roof = None
    if cand:
        name = max(cand)[1]
        e = kernels[name]
        roof = {"kernel": name, "bound": "hbm", "achieved": e["achieved_gbs"], "peak": hbm, "unit": "GB/s",
                "frac": e["frac_of_hbm"], "traffic": traffic.get(name), "avg_launch_ms": e["avg_ms"],
                "alg_bytes_per_launch": e["alg_bytes_per_launch"],
                "share_of_step": round(kt[name][1] / sum(v[1] for v in kt.values()), 3),
                "peak_kind": pk_kind + " (MEASURED_PEAKS.json hbm_gbs)",
                "how": "CUDA events around every launch on its stream, %d steps with one encoder in flight" % args.steps}

    # single-GPU side measurements (config 2 / config 3 kernels, decode): N = 1 only
    extra = extra_measurements(lib, api, hbm) if world == 1 else {"note": "side measurements run at N=1 only"}

    # ---------------- CPU baseline: the reference's own code on this box's host cores --------------

    # reference on the host: all cores of the box (the GPU arm's NUMA binding is lifted for it), one
    # frame per concurrent call, the same concurrency rule as `--impl reference`
    ncpu_all = os.cpu_count() or 1
    try:
        os.sched_setaffinity(0, range(ncpu_all))
    except OSError:
        pass
    if world == 1:
        cpu = cpu_baseline(frames, reps=2)   # two frames per host thread back to back, like the reference arm
    else:
        cpu = {"value": None, "unit": "MPix/s", "cores": 0, "kind": "reference", "sample": "timed at N=1 only"}

    line = {
        "metric": "MPix/s encode(API-1) at 4K",
        "value": round(value, 1), "unit": "MPix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(t_res / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "api1_encode_3840x2160_p010hlg_bt2100+yuv420_bt709", "frames_per_gpu_per_step": F, "host_buffers": "pinned",
                   "cpu_affinity": affinity, "encoder_slots": slots_n, "quality": 95, "gainmap": "multichannel scale 1 two-pass",
                   "l2_policy": "inputs larger than L2 (%d MB of frames per step, distinct per frame)" % (in_bytes >> 20),
                   "timing": "wall clock between device-wide synchronisations around exactly K steps (host threads walk the K steps "
                             "back to back, no join between steps), max over ranks; "
                             "per-kernel times from CUDA events on the launching streams"},
        "e2e": {"value": round(e2e_value, 1), "unit": "MPix/s", "h2d_bytes_per_step": int(in_bytes),
                "d2h_bytes_per_step": int(sum(e2e_out)), "ms_per_step": round(t_e2e / args.steps * 1e3, 3),
                "h2d_achieved_gbs": round(world * in_bytes / (t_e2e / args.steps) / 1e9, 1),
                "h2d_achieved_gbs_per_gpu": round(in_bytes / (t_e2e / args.steps) / 1e9, 1), "pcie_probe": pcie,
                "frac_of_h2d_probe": (round(world * in_bytes / (t_e2e / args.steps) / 1e9 / pcie["h2d_gbs_sum"], 3)
                                                 if world > 1 and pcie.get("h2d_gbs_sum") else
                                                 (round(in_bytes / (t_e2e / args.steps) / 1e9 / pcie["h2d_gbs"], 3) if pcie.get("h2d_gbs") else None)),
                "bound": "pcie h2d: 37.3 MB of raw pixels enter per 4K frame, 2.3 MB of JPEG/R leave"},
        "decode": {"metric": "MPix/s decode 8K JPEG/R -> RGBA half float", "e2e": {"value": round(dec_value, 1), "unit": "MPix/s",
                   "h2d_bytes_per_image": len(data8), "d2h_bytes_per_image": W8K * H8K * 8,
                   "d2h_achieved_gbs": round(dec_value * 8e6 / 1e9 / world, 1)},
                   "images": world * dec_handles * dec_per, "handles_per_gpu": dec_handles,
                   "cpu_baseline": (cpu_decode_baseline(data8, W8K, H8K) if world == 1 else None),
                   "how": "uhdr_dec_set_image + uhdr_decode + uhdr_get_decoded_image through the C ABI, compressed stream and "
                          "pixels in host memory, wall clock between device-wide synchronisations, max over ranks"},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "roofline": roof,
        "kernels": kernels,
        "cpu_baseline": cpu,
        "extra": extra,
        "stream_bytes_per_frame": int(sum(out_bytes) / max(1, F)),
        "stream_bytes_per_frame_e2e": int(sum(e2e_out) / max(1, F)),
        "resident_equals_e2e_streams": [int(x) for x in out_bytes] == [int(x) for x in e2e_out],
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def stream_bytes(lib, handle):
    o = lib.uhdr_get_encoded_stream(handle).contents
    return C.string_at(o.data, o.data_sz)


def dump_outputs(out_dir, streams, decoded):
    """--dump-outputs: what the timed paths returned in their last step on rank 0, as .npy files (float32 /
    float64) that two builds can be compared with, at most 48 MB in all:
      stream_length.npy         float64 (F,)       bytes of each frame's JPEG/R file (API-1 encode arm)
      stream_bytes_sample.npy   float32 (F, S)     byte values, S = min(2^18, 2^23 / F): the first min(4096, S)
                                                   bytes of each file (headers, metadata), then offsets drawn
                                                   uniformly from the rest with numpy RandomState(frame index),
                                                   in increasing order
      decode_8k_rgba_sample.npy float32 (2^20, 4)  RGBA half-float pixels of the 8K decode arm, at 2^20 pixel
                                                   indices drawn with RandomState(0), in increasing order"""
    os.makedirs(out_dir, exist_ok=True)
    n = len(streams)
    per = max(1, min(1 << 18, (32 << 20) // 4 // max(1, n)))
    head = min(4096, per)
    sample = np.zeros((n, per), np.float32)
    for i, s in enumerate(streams):
        b = np.frombuffer(s, np.uint8)
        k = min(head, b.size)
        rest = np.sort(np.random.RandomState(i).randint(k, max(k + 1, b.size), per - k)) if b.size > k else np.zeros(per - k, np.int64)
        idx = np.concatenate([np.arange(k), rest]) if b.size else np.zeros(per, np.int64)
        sample[i] = b[idx] if b.size else 0
    np.save(os.path.join(out_dir, "stream_length.npy"), np.array([len(s) for s in streams], np.float64))
    np.save(os.path.join(out_dir, "stream_bytes_sample.npy"), sample)
    w, h = decoded.w, decoded.h
    px = np.ctypeslib.as_array(C.cast(decoded.planes[0], C.POINTER(C.c_uint16)), (h, decoded.stride[0] * 4))[:, :w * 4]
    flat = px.reshape(h * w, 4)
    pick = np.sort(np.random.RandomState(0).randint(0, h * w, 1 << 20))
    np.save(os.path.join(out_dir, "decode_8k_rgba_sample.npy"), flat[pick].view(np.float16).astype(np.float32))


def apply_8k(lib, hbm, iters=6):
    """applyGainMap kernel at 7680x4320 (config 3 geometry), CUDA-event time per launch"""
    import uhdr_testlib as T
    out = {}
    gpu = T.Gpu()
    # applyGainMap at 8K: RGBA8888 map, scale 1 (13.5 B/px).  Two contents: "natural" (smooth +
    # texture, like the encode frames) and uniform noise (worst case for the table gathers)
    md = A.GainmapMetadata()
    for i, (mx, mn) in enumerate(((65.1, 4.9e-5), (845.9, 2.7e-3), (1283.8, 4.9e-5))):
        md.max_content_boost[i], md.min_content_boost[i], md.gamma[i] = mx, mn, 1.0
        md.offset_sdr[i] = md.offset_hdr[i] = 1e-7
    md.hdr_capacity_min, md.hdr_capacity_max, md.use_base_cg = 1.0, 4.926108, 0
    lib.uhdr_b200_set_kernel_timing(1)
    for content in ("natural", "noise"):
        if content == "noise":
            sb = T.make_yuv420(W8K, H8K, "noise")
            gm = np.random.RandomState(7).randint(0, 256, (H8K, W8K, 4)).astype(np.uint8)
        else:
            _p, sb = make_frame(W8K, H8K, 5)
            yy, xx = np.mgrid[0:H8K, 0:W8K].astype(np.float32)
            g0 = 128 + 90 * np.sin(xx / 301.0) * np.cos(yy / 257.0) + np.random.RandomState(3).randn(H8K, W8K) * 2
            gm = np.stack([g0, g0 * 0.9 + 10, g0 * 0.8 + 20, np.full_like(g0, 255)], -1).clip(0, 255).astype(np.uint8)
            del yy, xx, g0, _p
        sdr, k2 = A.yuv420_image(sb, W8K, H8K, A.CG_BT709)
        gi = T.gm_image(gm, A.CG_BT2100)
        for _ in range(3):  # warm-up: module load, arena growth, clocks
            gpu.apply(sdr, gi, md, A.CT_LINEAR)
        kernel_report(lib)
        for _ in range(iters):
            gpu.apply(sdr, gi, md, A.CT_LINEAR)
        kt = kernel_report(lib)
        if "apply_gainmap" in kt:
            cnt, ms = kt["apply_gainmap"][:2]
            mn_ms, mx_ms = (kt["apply_gainmap"] + (None, None))[2:4]
            avg = ms / cnt
            alg = 13.5 * W8K * H8K
            out["apply_gainmap_8k_" + content] = {
                "avg_launch_ms": round(avg, 4), "min_launch_ms": mn_ms, "max_launch_ms": mx_ms, "launches": cnt, "mpix_s": round(W8K * H8K / 1e6 / (avg * 1e-3), 1),
                "roofline": {"bound": "hbm", "achieved": round(alg / (avg * 1e-3) / 1e9, 1), "peak": hbm, "unit": "GB/s",
                             "frac": round(alg / (avg * 1e-3) / 1e9 / hbm, 4), "alg_bytes_per_launch": int(alg)}}
        del sb, gm
    lib.uhdr_b200_set_kernel_timing(0)
    return out


def extra_measurements(lib, api, hbm):
    """config 3 (8K decode -> RGBA half float) and config 2 (4K API-0), device timings of the
    kernels named by the north star; small step counts, not the headline."""
    import uhdr_testlib as T
    out = {}
    try:
        out.update(apply_8k(lib, hbm))
        lib.uhdr_b200_set_kernel_timing(1)
        # API-0 4K through the C API (resident inputs)
        p010, _ = make_frame(W4K, H4K, 99)
        hdr, _k = A.p010_image(p010, W4K, H4K, A.CG_BT2100, A.CT_HLG, A.CR_LIMITED)
        sl = EncoderSlot(lib)
        sl.set_inputs(hdr, None)
        for _ in range(3):
            sl.encode()
            sl.rearm()
        kernel_report(lib)
        t0 = time.perf_counter()
        n = 5
        for _ in range(n):
            sl.rearm()
            sl.encode()
        dt = (time.perf_counter() - t0) / n
        kt = kernel_report(lib)
        out["api0_encode_4k"] = {"mpix_s_resident_1slot": round(MPIX_4K / dt, 1), "ms_per_frame": round(dt * 1e3, 3),
                                 "kernels_avg_ms": {k: round(v[1] / v[0], 4) for k, v in kt.items()}}
        lib.uhdr_b200_set_kernel_timing(0)
        # config 3 end to end: uhdr_decode of a JPEG/R (multichannel map, scale 1) to RGBA half float
        # through the drop-in C ABI: compressed stream in host memory -> pixels in host memory.  Entropy
        # decoding, IDCT, applyGainMap all on the device; per call a new decoder handle, like the
        # reference's examples do.
        lib.uhdr_b200_entropy_decoder_stats.restype = None
        for tag, (w, h) in (("4k", (W4K, H4K)), ("8k", (W8K, H8K))):
            p8, y8 = make_frame(w, h, 7)
            h8, s8, _k8 = frame_descs(p8, y8, w, h)
            data = api.encode(h8, s8)

            def timed_decode(L, n, data=data, w=w, sdr_out=False):
                buf = np.frombuffer(data, np.uint8).copy()
                ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
                ts = []
                for _ in range(n):
                    dec = C.c_void_p(L.uhdr_create_decoder())
                    t0 = time.perf_counter()
                    assert L.uhdr_dec_set_image(dec, C.byref(ci)).error_code == 0
                    if sdr_out:   # the decoder's UHDR_CT_SRGB leg: base image only, 32bppRGBA8888
                        L.uhdr_dec_set_out_img_format.restype = A.ErrorInfo
                        L.uhdr_dec_set_out_color_transfer.restype = A.ErrorInfo
                        assert L.uhdr_dec_set_out_img_format(dec, A.FMT_RGBA8888).error_code == 0
                        assert L.uhdr_dec_set_out_color_transfer(dec, A.CT_SRGB).error_code == 0
                    e = L.uhdr_decode(dec)
                    assert e.error_code == 0, e.detail
                    assert L.uhdr_get_decoded_image(dec).contents.w == w
                    ts.append(time.perf_counter() - t0)
                    L.uhdr_release_decoder(dec)
                return min(ts), sorted(ts)[len(ts) // 2]
            st0 = (C.c_ulonglong * 3)()
            st1 = (C.c_ulonglong * 3)()
            lib.uhdr_b200_entropy_decoder_stats(st0)
            dt, med = timed_decode(lib, 6)
            lib.uhdr_b200_entropy_decoder_stats(st1)
            key = "decode_%s_e2e" % tag
            out[key] = {"ms": round(dt * 1e3, 2), "ms_median": round(med * 1e3, 2), "mpix_s": round(w * h / 1e6 / dt, 1),
                        "stream_bytes": len(data), "d2h_bytes": w * h * 8,
                        "entropy_decoder": {"device_scans": int(st1[0] - st0[0]), "handed_to_host": int(st1[1] - st0[1]),
                                            "relaxation_rounds_last": int(st1[2])},
                        "note": "uhdr_dec_set_image + uhdr_decode + uhdr_get_decoded_image through the C ABI, best of 6; "
                                "output 64bppRGBAHalfFloat in handle-owned pinned memory"}
            dts, meds = timed_decode(lib, 4, sdr_out=True)
            out[key]["sdr_output_ct_srgb_rgba8888"] = {"ms": round(dts * 1e3, 2), "ms_median": round(meds * 1e3, 2),
                                                       "mpix_s": round(w * h / 1e6 / dts, 1), "d2h_bytes": w * h * 4}
            # several decoder handles in flight, one host thread each, every handle reused through
            # uhdr_reset_decoder (its arenas stay sized): stream in / pixels out of different images overlap
            nthr, per = 4, 6
            bar = threading.Barrier(nthr + 1)

            def worker(data=data, w=w):
                buf = np.frombuffer(data, np.uint8).copy()
                ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)
                dec = C.c_void_p(lib.uhdr_create_decoder())
                for it in range(2 + per):
                    if it == 2:
                        bar.wait()
                    lib.uhdr_reset_decoder(dec)
                    assert lib.uhdr_dec_set_image(dec, C.byref(ci)).error_code == 0
                    e = lib.uhdr_decode(dec)
                    assert e.error_code == 0, e.detail
                    assert lib.uhdr_get_decoded_image(dec).contents.w == w
                lib.uhdr_release_decoder(dec)
            ths = [threading.Thread(target=worker) for _ in range(nthr)]
            for t in ths:
                t.start()
            bar.wait()
            t0 = time.perf_counter()
            for t in ths:
                t.join()
            dtb = time.perf_counter() - t0
            out[key]["throughput_mpix_s_4_handles"] = round(nthr * per * w * h / 1e6 / dtb, 1)
            if T.have_ref():
                rapi, rlib = load_api(T.REF_SO)
                dtr, _m = timed_decode(rlib, 1)
                out[key]["cpu_reference_ms"] = round(dtr * 1e3, 1)
                out[key]["cpu_reference_mpix_s"] = round(w * h / 1e6 / dtr, 1)
            del p8, y8, data
    except Exception as e:  # noqa: BLE001
        out["error"] = repr(e)
    # config 5: generateGainMap (two-pass, multichannel, scale 1) at 4K over transfer x HDR gamut, SDR
    # intent BT.709: kernel times of pass 1 + affine pass by CUDA events.  The gamut decides which side
    # carries the 3x3 conversion (jpegr.cpp:607-638), the transfer which inverse-OETF table is staged.
    try:
        gpu = T.Gpu()
        p010, yuv = make_frame(W4K, H4K, 11)
        sdr, _ks = A.yuv420_image(yuv, W4K, H4K, A.CG_BT709)
        lib.uhdr_b200_set_kernel_timing(1)
        def sweep_over(cfg, names):
            res = {}
            for ct_name, ct in (("hlg", A.CT_HLG), ("pq", A.CT_PQ), ("srgb", A.CT_SRGB)):
                for cg_name, cg in (("bt709", A.CG_BT709), ("p3", A.CG_P3), ("bt2100", A.CG_BT2100)):
                    hdr, _kh = A.p010_image(p010, W4K, H4K, cg, ct, A.CR_LIMITED)
                    gpu.generate(sdr, hdr, cfg)
                    kernel_report(lib)
                    for _ in range(3):
                        gpu.generate(sdr, hdr, cfg)
                    kt = kernel_report(lib)
                    ms = sum(kt[k][1] / kt[k][0] for k in names if k in kt)
                    res[ct_name + "_" + cg_name] = {"kernels_ms": round(ms, 4), "mpix_s": round(MPIX_4K / (ms * 1e-3), 1)}
            return res
        # sRGB: not an encoder input (uhdr_enc_set_raw_image refuses it) but a valid JpegR::generateGainMap transfer
        sweep = sweep_over(None, ("gainmap_pass1", "gainmap_affine"))
        # JpegR's own defaults (ultrahdrcommon.h:450-457): map scale 4, one channel; both presets
        out["config5_generate_gainmap_4k_scale4_1ch_twopass"] = sweep_over(
            A.default_gm_config(scale_factor=4, multichannel=0, preset=1), ("gainmap_pass1", "gainmap_affine"))
        out["config5_generate_gainmap_4k_scale4_1ch_realtime"] = sweep_over(
            A.default_gm_config(scale_factor=4, multichannel=0, preset=0), ("gainmap_onepass",))
        lib.uhdr_b200_set_kernel_timing(0)
        out["config5_generate_gainmap_4k"] = sweep
    except Exception as e:  # noqa: BLE001
        out["config5_error"] = repr(e)
    return out


def ref_jpeg_note():
    import uhdr_testlib as T
    if T.ref_is_turbo():
        return "reference sources incl. its own jpeg{en,de}coderhelper.cpp on the real libjpeg-turbo (Pillow's 3.1.x binary, SIMD)"
    return "reference sources, JPEG through oracle/jpeg_oracle.c (scalar) because no libjpeg-turbo binary was found"


def ref_concurrency(gb_per_call):
    """concurrent reference calls: one per host thread (measured here: throughput still rises up to
    one call per hardware thread although each call also spawns the reference's own <=4 workers),
    bounded by free memory"""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    conc = ncpu
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                conc = min(conc, max(1, int(int(ln.split()[1]) / 1048576 * 0.6 / gb_per_call)))
    except OSError:
        pass
    return max(1, conc), ncpu


def cpu_baseline(frames, reps=1):
    """reference CPU path (oracle/_ref) on the host cores: API-1 4K encode of a bounded sample."""
    import uhdr_testlib as T
    if not T.have_ref():
        return {"value": None, "unit": "MPix/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref missing"}
    api, lib = load_api(T.REF_SO)
    conc, ncpu = ref_concurrency(0.5)
    descs = [frame_descs(p, y, W4K, H4K) for (p, y) in frames]
    api.encode(descs[0][0], descs[0][1])  # first call builds the reference's static LUTs
    t0 = time.perf_counter()
    done = [0] * conc

    def work(i):
        for r in range(reps):
            api.encode(descs[i % len(descs)][0], descs[i % len(descs)][1])
            done[i] += 1
    run_threads(conc, work)
    dt = time.perf_counter() - t0
    n = sum(done)
    return {"value": round(n * MPIX_4K / dt, 2), "unit": "MPix/s", "cores": ncpu, "kind": "reference",
            "sample": "%d x 4K API-1 uhdr_encode calls, %d concurrent on %d host threads, %.1f s; %s" % (n, conc, ncpu, dt, ref_jpeg_note()),
            "host_cpus": ncpu}


def cpu_decode_baseline(data, w, h, reps=1):
    """reference uhdr_decode (-> RGBA half float) of one JPEG/R, one call per host thread"""
    import uhdr_testlib as T
    if not T.have_ref():
        return None
    api, lib = load_api(T.REF_SO)
    conc, ncpu = ref_concurrency(w * h * 40 / 1e9)
    buf = np.frombuffer(data, np.uint8).copy()
    ci = A.CompressedImage(buf.ctypes.data, len(data), len(data), -1, -1, -1)

    def one():
        dec = C.c_void_p(lib.uhdr_create_decoder())
        assert lib.uhdr_dec_set_image(dec, C.byref(ci)).error_code == 0
        e = lib.uhdr_decode(dec)
        assert e.error_code == 0, e.detail
        assert lib.uhdr_get_decoded_image(dec).contents.w == w
        lib.uhdr_release_decoder(dec)
    t0 = time.perf_counter()
    one()
    t_single = time.perf_counter() - t0
    t0 = time.perf_counter()
    run_threads(conc, lambda i: [one() for _ in range(reps)])
    dt = time.perf_counter() - t0
    return {"value": round(conc * reps * w * h / 1e6 / dt, 2), "unit": "MPix/s", "cores": ncpu, "kind": "reference",
            "single_call_ms": round(t_single * 1e3, 1),
            "sample": "%d uhdr_decode calls of one %dx%d JPEG/R -> RGBA half float, %d concurrent on %d host threads, %.1f s; %s"
                      % (conc * reps, w, h, conc, ncpu, dt, ref_jpeg_note())}


def bench_reference(args, rank, world):
    if rank != 0:
        return
    import uhdr_testlib as T
    T.ensure_oracle_built()
    if not T.have_ref():
        emit({"impl": "reference", "unavailable": "oracle/_ref/libuhdr_ref.so not built (needs /root/reference at build time)"})
        return
    api, lib = load_api(T.REF_SO)
    conc, ncpu = ref_concurrency(0.5)
    frames = [make_frame(W4K, H4K, i) for i in range(min(conc, 8))]
    descs = [frame_descs(p, y, W4K, H4K) for (p, y) in frames]
    per_step = conc   # a step = one 4K frame per concurrent call: the bounded sample of the GPU arm's 32-frame batch

    def step():
        run_threads(conc, lambda i: api.encode(descs[i % len(descs)][0], descs[i % len(descs)][1]))
    t0 = time.perf_counter()
    step()            # also builds the reference's static LUTs
    t_first = time.perf_counter() - t0
    # keep the whole run within a few minutes whatever K and W the driver passes
    steps, warmup = args.steps, args.warmup
    budget = 150.0
    if (steps + warmup) * t_first > budget:
        warmup = min(warmup, 1)
        steps = max(1, min(steps, int(budget / t_first) - warmup))
    for _ in range(max(0, warmup - 1)):
        step()
    # same rule as the GPU arm: the host threads walk the K steps back to back, no join between steps (a join
    # would make every step wait for its slowest call, which costs the 128-thread arm more than the GPU arm)
    t0 = time.perf_counter()
    run_threads(conc, lambda i: [api.encode(descs[i % len(descs)][0], descs[i % len(descs)][1]) for _ in range(steps)])
    dt = time.perf_counter() - t0
    v = per_step * steps * MPIX_4K / dt
    sample = "%d concurrent 4K API-1 uhdr_encode calls per step on %d host threads; %s" % (conc, ncpu, ref_jpeg_note())
    # decode arm of the metric (config 3): 8K JPEG/R written by the reference itself, all host threads
    decode = None
    try:
        p8, y8 = make_frame(W8K, H8K, 7)
        h8, s8, _k8 = frame_descs(p8, y8, W8K, H8K)
        data8 = api.encode(h8, s8)
        del p8, y8
        decode = cpu_decode_baseline(data8, W8K, H8K)
        decode["metric"] = "MPix/s decode 8K JPEG/R -> RGBA half float"
    except Exception as e:  # noqa: BLE001
        decode = {"error": repr(e)}
    emit({
        "impl": "reference", "metric": "MPix/s encode(API-1) at 4K", "value": round(v, 2), "unit": "MPix/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": round(dt / steps * 1e3, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "api1_encode_3840x2160_p010hlg_bt2100+yuv420_bt709", "frames_per_step": per_step,
                   "steps_requested": args.steps, "warmup_requested": args.warmup},
        "cpu_baseline": {"value": round(v, 2), "unit": "MPix/s", "cores": ncpu, "kind": "reference", "sample": sample},
        "e2e": {"value": round(v, 2), "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "decode": decode,
    })


_REAL_STDOUT = None


def emit(obj):
    """the one JSON line, on the process's real stdout"""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=32, help="4K frames per GPU per step (config 4: 32 per GPU)")
    ap.add_argument("--slots", type=int, default=8, help="concurrent encoder handles (host threads) per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they returned in the last step to DIR/*.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    # stdout must carry exactly one JSON line: while the bench runs, file descriptor 1 points at
    # stderr (NCCL and other libraries print banners to stdout); emit() switches it back
    sys.stdout.flush()
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        bench_reference(args, rank, world)
    else:
        if args.warmup < 3:
            args.warmup = 3
        bench_b200(args, rank, world)


if __name__ == "__main__":
    main()
