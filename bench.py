#!/usr/bin/env python
"""bench.py -- Mpixels/s of baseline 4:2:0 batch decode on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload hd1024|uhd] [--dump-outputs DIR]

A "step" = one pass of the hot path (prescan -> entropy -> stitch -> fused IDCT+colour) over
one batch of synthetic JPEGs.  N=1 workload = BASELINE.json configs[1]: 1024 x 1920x1080
4:2:0 q75 -> RGB8888.  `value` = source megapixels/s with compressed inputs resident in HBM
and pixels left in HBM; `e2e` = the same metric through the public C ABI with pinned HOST
buffers on both sides (header parse + H2D + kernels + D2H inside the timed region).
`--impl reference` times the unmodified reference (oracle/_ref, SSE2 build) on all host cores.
One JSON line on stdout (rank 0).  `--dump-outputs DIR` also writes what the last timed step decoded (rank 0's batch) as
.npy files, so that two builds can be compared output for output: the inputs are the same seeded images on every run.
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
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from as it found it

WORKLOADS = {
    # name: (n_images, w, h, quality, pixel_type_name, algorithmic bytes per source pixel for the fused kernel)
    "hd1024": dict(n=1024, w=1920, h=1080, q=75, pt="RGB8888", bpp_out=4, coef_bpp=3,
                   desc="1024 x 1920x1080 4:2:0 q75 -> RGB8888 (BASELINE.json configs[1])"),
    "uhd": dict(n=512, w=3840, h=2160, q=85, pt="RGB565_LITTLE_ENDIAN", bpp_out=2, coef_bpp=3,
                desc="512 x 3840x2160 4:2:0 q85 -> RGB565 per GPU (BASELINE.json configs[2] shape, per-GPU slice)"),
    "dither": dict(n=256, w=2048, h=1536, q=75, pt="ONE_BIT_DITHERED", bpp_out=0.125, coef_bpp=2, gray=True,
                   desc="256 x 2048x1536 1-component q75 -> 1-bpp Floyd-Steinberg (BASELINE.json configs[4] shape)"),
    "dither1024": dict(n=1024, w=2048, h=1536, q=75, pt="ONE_BIT_DITHERED", bpp_out=0.125, coef_bpp=2, gray=True,
                       desc="1024 x 2048x1536 1-component q75 -> 1-bpp Floyd-Steinberg (configs[4] shape at the batch size of configs[1]: below ~512 images "
                            "jdk_dither is bound by one image's row-to-row dependency chain, not by throughput)"),
    "hd_norst": dict(n=1024, w=1920, h=1080, q=75, pt="RGB8888", bpp_out=4, coef_bpp=3, restart_rows=0,
                     desc="1024 x 1920x1080 4:2:0 q75 WITHOUT restart markers -> RGB8888 (SURVEY 8(f)2: chunk-parallel entropy decode)"),
    "uhd_quarter": dict(n=512, w=3840, h=2160, q=85, pt="RGB565_LITTLE_ENDIAN", bpp_out=2.0 / 16, coef_bpp=0.1875, opt=4, kernel="jdk_scaled",
                        desc="512 x 3840x2160 4:2:0 q85 -> RGB565 at JPEG_SCALE_QUARTER (BASELINE.json configs[3]); MP = source pixels"),
    "uhd_eighth": dict(n=512, w=3840, h=2160, q=85, pt="RGB565_LITTLE_ENDIAN", bpp_out=2.0 / 64, coef_bpp=0.046875, opt=8, kernel="jdk_scaled",
                       desc="512 x 3840x2160 4:2:0 q85 -> RGB565 at JPEG_SCALE_EIGHTH (BASELINE.json configs[3]); MP = source pixels"),
    "dither444": dict(n=256, w=2048, h=1536, q=75, pt="ONE_BIT_DITHERED", bpp_out=0.125, coef_bpp=6, subsampling="4:4:4",
                      desc="256 x 2048x1536 4:4:4 colour q75 -> 1-bpp Floyd-Steinberg (BASELINE.json configs[4], colour variant)"),
    "uhd10k": dict(n=1250, w=3840, h=2160, q=85, pt="RGB565_LITTLE_ENDIAN", bpp_out=2, coef_bpp=3, unique=32, verify_all=True,
                   desc="BASELINE.json configs[2]: 10 000 x 3840x2160 4:2:0 q85 -> RGB565 sharded over 8 GPUs = 1250 images per GPU "
                        "(32 unique seeds per GPU = 256 over 8 ranks, cycled); every image's device-resident pixels are verified "
                        "by digest against the reference"),
    "tiny": dict(n=16, w=640, h=480, q=75, pt="RGB8888", bpp_out=4, coef_bpp=3, desc="16 x 640x480 (smoke)"),
}


def host_cpu_facts():
    """What the process may actually use (the judge's round-1 finding: os.cpu_count() said 128 on a lease with ~16)."""
    facts = {"os_cpu_count": os.cpu_count()}
    try:
        facts["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        facts["affinity"] = None
    quota = None
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt and txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    facts["cgroup_cpu_quota"] = quota
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                facts["model"] = line.split(":", 1)[1].strip()
                break
    except Exception:
        facts["model"] = None
    try:
        facts["numa_nodes"] = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
    except Exception:
        facts["numa_nodes"] = None
    usable = facts["affinity"] or facts["os_cpu_count"] or 1
    if quota:
        usable = max(1, min(usable, int(quota + 0.5)))
    facts["usable"] = usable
    return facts


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this workload's kernel
    instance (profiles/roofline_traffic.json: {workload: {"bytes": dram read + write, "kernel": instance, "from": summary file}});
    None when no capture of this build's instance is committed."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            e = json.load(open(p)).get(workload)
            if isinstance(e, dict):
                return e.get("bytes"), e
            return None, None
        except Exception:
            return None, None
    return None, None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line): an NVML polling
    thread (5 ms period; the timed region of a short run is only tens of milliseconds), nvidia-smi -lms as the fallback."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, gpu_index):
        self.rows = []          # (time, sm_mhz, max_mhz, reasons bitmask)
        self.gpu = gpu_index
        self.stop_flag = False
        self.t = None
        self.mode = None

    def _nvml_loop(self, pynvml, h, mx):
        while not self.stop_flag:
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.time(), float(sm), float(mx), int(rs)))
            except Exception:
                pass
            time.sleep(0.005)

    def _smi_loop(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                bits = 0
                for (bit, _), v in zip(self.REASONS, f[3:7]):
                    if v.lower().startswith("active"):
                        bits |= bit
                self.rows.append((time.time(), float(f[0]), float(f[1]), bits))
            except Exception:
                continue

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical GPUs: honour CUDA_VISIBLE_DEVICES when it is a list of indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.gpu
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.mode = "nvml"
            self.t = threading.Thread(target=self._nvml_loop, args=(pynvml, h, mx), daemon=True)
            self.t.start()
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.mode = "nvidia-smi"
            self.t = threading.Thread(target=self._smi_loop, daemon=True)
            self.t.start()
        except Exception:
            self.mode = None

    def stop(self, t0, t1):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        if self.mode == "nvidia-smi":
            time.sleep(0.1)
            self.proc.terminate()
        self.stop_flag = True
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        note = None
        if not inside and self.rows:   # region shorter than one sample: nearest samples
            inside = sorted(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:3]
            note = "no sample inside the timed region; nearest samples used"
        sm = [r[1] for r in inside]
        bits = 0
        for r in inside:
            bits |= r[3]
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": inside[0][2] if inside else None,
               "reasons": [name for bit, name in self.REASONS if bits & bit], "samples": len(sm), "source": self.mode}
        if note:
            out["note"] = note
        return out


def make_images(wl, rank, unique):
    from tests import synth
    # every rank generates its own images at the same time: share the host cores between the ranks
    world = max(1, int(os.environ.get("WORLD_SIZE", "1")))
    workers = max(2, min(64, host_cpu_facts()["usable"] // world))
    jp = synth.synth_set(unique, wl["w"], wl["h"], quality=wl["q"], seed0=rank * unique, gray=wl.get("gray", False),
                         restart_rows=wl.get("restart_rows", 1), subsampling=wl.get("subsampling", "4:2:0"), workers=workers)
    return jp


def cpu_reference_run(wl, jpegs, pixel_type, n_sample, threads, passes=3):
    """Times the unmodified reference (oracle/_ref SSE2 build), framebuffer mode, `threads` workers."""
    from oracle import refdrv
    ref = refdrv.Ref("sse")
    datas = [jpegs[i % len(jpegs)] for i in range(n_sample)]
    rows = ((wl["h"] + 15) // 16) * 16 + 16
    bypp = max(1, int(wl["bpp_out"]))
    # one framebuffer per worker slot is enough for timing (image i -> worker i % threads writes fbs[i])
    pool = [np.empty(rows * wl["w"] * bypp + 4096, dtype=np.uint8) for _ in range(min(threads, n_sample))]
    fbs = [pool[i % len(pool)] for i in range(n_sample)]
    best = None
    for _ in range(passes):
        fails, secs = ref.decode_batch(datas, pixel_type, wl.get("opt", 0), threads, fbs)
        if fails:
            raise RuntimeError("reference failed on %d images" % fails)
        best = secs if best is None else min(best, secs)
    mp = n_sample * wl["w"] * wl["h"] / 1e6
    return mp / best, best


def dump_outputs(out_dir, b, st, n_img, oh0, row_bytes):
    """The last timed step's results as a caller of the batch would read them: per image its status and the CRC-32 of its
    pixels (rows x bytes that hold image pixels), and the pixel bytes of a fixed seeded sample of up to 8 images at a fixed
    seeded sample of up to 2^20 byte offsets.  float64 / float32 .npy files, about 40 MB at most."""
    import zlib
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    img_bytes = oh0 * row_bytes
    pick = np.sort(rng.choice(n_img, size=min(8, n_img), replace=False))
    offs = np.sort(rng.choice(img_bytes, size=min(1 << 20, img_bytes), replace=False))
    crc = np.zeros(n_img, dtype=np.float64)
    pixels = np.zeros((len(pick), len(offs)), dtype=np.float32)
    for i in range(n_img):
        img = np.ascontiguousarray(b.read_output(i)[:oh0, :row_bytes]).reshape(-1)
        crc[i] = zlib.crc32(img)
        k = np.searchsorted(pick, i)
        if k < len(pick) and pick[k] == i:
            pixels[k] = img[offs]
    np.save(os.path.join(out_dir, "status.npy"), np.asarray(st, dtype=np.float64))
    np.save(os.path.join(out_dir, "crc32.npy"), crc)
    np.save(os.path.join(out_dir, "pixels.npy"), pixels)
    np.save(os.path.join(out_dir, "pixel_images.npy"), pick.astype(np.float64))
    np.save(os.path.join(out_dir, "pixel_offsets.npy"), offs.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="hd1024")
    ap.add_argument("--unique", type=int, default=64, help="unique synthetic images per rank (cycled to the batch size)")
    ap.add_argument("--images", type=int, default=0, help="development aid: override the workload's images per GPU (the line's config says so)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--pipelined", action="store_true", help="also time the steps with two resident batches in flight")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's decoded outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    W = max(args.warmup, 0)
    K = args.steps
    cpu_facts = host_cpu_facts()
    threads = cpu_facts["usable"]
    n_img = args.images if args.images > 0 else wl["n"]
    if "unique" in wl:
        args.unique = wl["unique"]
    mp_per_step_rank = n_img * wl["w"] * wl["h"] / 1e6
    config = {"workload": wl["desc"], "images_per_gpu": n_img, "width": wl["w"], "height": wl["h"],
              "quality": wl["q"], "subsampling": "4:2:0", "restart_interval": "1 MCU row",
              "pixel_type": wl["pt"], "arith_mode": "SSE2-build parity", "parallelism": "images sharded, dp%d" % world,
              "l2_policy": "inputs_exceed_l2 (per step: %.0f MB compressed + %.1f GB pixels >> 126 MB L2)" % (
                  n_img * 0.29 if args.workload == "hd1024" else n_img * 1.6, n_img * wl["w"] * wl["h"] * wl["bpp_out"] / 1e9),
              "value_excludes": "H2D of the compressed bytes (resident in HBM before the timed region; its time is stages_ms.h2d) and any D2H; e2e includes both"}

    import jpegdec_b200 as J
    pixel_type = getattr(J, wl["pt"])

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        from oracle import refdrv
        if not refdrv.available("sse"):
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libjpegdec_ref_sse.so not built"}))
            return 0
        jpegs = make_images(wl, 0, min(args.unique, 32))
        n_sample = max(threads * 4, 128)
        for _ in range(W):
            cpu_reference_run(wl, jpegs, pixel_type, max(threads, 16), threads, passes=1)
        t_total, mp_total = 0.0, 0.0
        for _ in range(K):
            mps, secs = cpu_reference_run(wl, jpegs, pixel_type, n_sample, threads, passes=1)
            t_total += secs
            mp_total += n_sample * wl["w"] * wl["h"] / 1e6
        v = mp_total / t_total
        sample = "%d images per step (%d unique, cycled), framebuffer mode, openRAM..close per image" % (n_sample, len(jpegs))
        print(json.dumps({
            "impl": "reference", "metric": "Mpixels/sec baseline 4:2:0 decode (batch)", "value": v, "unit": "Mpixels/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * t_total / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int16/int32 (SSE2 build)", "data": "synthetic",
            "config": dict(config, note="reference CPU path, all host threads; each step is a bounded sample of the workload"),
            "cpu_baseline": {"value": v, "unit": "Mpixels/s", "cores": threads, "kind": "reference", "sample": sample, "host": cpu_facts},
            "e2e": {"value": v, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    unique = min(args.unique, n_img)
    jpegs = make_images(wl, rank, unique)
    ctx = J.Context(local_rank, J.JPEG_ARITH_SSE2)
    # pinned host buffers and the thread that drives the copies go next to this rank's GPU (two-socket hosts: GPU0-3 on
    # node 0, GPU4-7 on node 1); the CPU baseline below restores the full mask first
    full_affinity = os.sched_getaffinity(0)
    bound_cpus = 0 if os.environ.get("JPEGDEC_B200_NO_BIND") else ctx.bind_host_to_device()
    numa = {"gpu_node": ctx.numa_node(), "bound_cpus": bound_cpus}
    # shared Huffman/quant table blob: rank 0 exports, NCCL broadcast, every rank imports
    blob = torch.zeros(J.TABLE_BLOB_BYTES, dtype=torch.uint8, device="cuda")
    if rank == 0:
        blob.copy_(torch.from_numpy(ctx.export_tables(jpegs[0])))
    if world > 1:
        dist.broadcast(blob, src=0)
    ctx.set_shared_tables(blob.cpu().numpy())

    # pinned input blob: the batch's files back to back (16-byte aligned starts)
    sizes = [len(jpegs[i % unique]) for i in range(n_img)]
    offs, o = [], 0
    for s in sizes:
        offs.append(o)
        o += (s + 15) & ~15
    L = J.lib()
    in_ptr = L.JPEGB200_hostAlloc(o + 64)
    in_arr = np.ctypeslib.as_array(C.cast(in_ptr, C.POINTER(C.c_ubyte)), shape=(o + 64,))
    in_arr[:] = 0
    for i in range(n_img):
        in_arr[offs[i]:offs[i] + sizes[i]] = np.frombuffer(jpegs[i % unique], dtype=np.uint8)
    ptrs = [in_ptr + off for off in offs]

    # ---- device-resident throughput (`value`) ----
    opt = int(wl.get("opt", 0))
    b = J.Batch(ctx, ptrs, sizes, pixel_type, opt)
    b.alloc_device_output()
    b.upload()
    b.decode(J.JPEGB200_OUT_DEVICE); b.download(); st = b.wait()
    if any(st):
        raise SystemExit("decode failed: %s" % st[:8])
    for _ in range(max(W - 1, 0)):
        b.decode(J.JPEGB200_OUT_DEVICE); b.download(); b.wait()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.02)
    barrier()
    t0 = time.time()
    dev_ms, stage = 0.0, {k: 0.0 for k in J.TIMING_NAMES}
    launches = 0
    for _ in range(K):
        b.decode(J.JPEGB200_OUT_DEVICE); b.download(); st = b.wait()
        tm = b.timings()
        dev_ms += tm["total"]
        for k in stage:
            stage[k] += tm[k]
        launches += b.counters()["launches"]
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    cnt = b.counters()
    ms_step = max_over_ranks(dev_ms / K)
    wall_ms_step = max_over_ranks(1e3 * (t1 - t0) / K)
    value = world * mp_per_step_rank / (ms_step / 1e3)
    idct_ms = stage["idct"] / K
    entropy_ms = stage["entropy"] / K
    sh0 = {2: 1, 4: 2, 8: 3}.get(opt & 14, 0)
    ow0, oh0 = (wl["w"] + (1 << sh0) - 1) >> sh0, (wl["h"] + (1 << sh0) - 1) >> sh0
    row_bytes = (ow0 * J.bits_per_pixel(pixel_type) + 7) // 8     # bytes of a row that hold image pixels (dithered rows are MCU-padded)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, b, st, n_img, oh0, row_bytes)

    # ---- the same steps with TWO batches in flight (informational): step k+1's entropy kernel (latency bound, ~45 % of
    # the issue slots) runs beside step k's IDCT kernel on another stream.  Wall clock around 2K decodes, max over ranks. ----
    pipelined = None
    if args.pipelined and not wl.get("verify_all"):
        try:
            b2 = J.Batch(ctx, ptrs, sizes, pixel_type, opt)
            b2.alloc_device_output(); b2.upload()
            pair = (b, b2)
            b2.decode(J.JPEGB200_OUT_DEVICE); b2.download(); b2.wait()
            barrier()
            tp0 = time.time()
            for k2 in range(2 * K):
                x = pair[k2 & 1]
                if k2 >= 2:
                    x.wait()
                x.decode(J.JPEGB200_OUT_DEVICE); x.download()
            b.wait(); b2.wait()
            barrier()
            tp1 = time.time()
            p_ms = max_over_ranks(1e3 * (tp1 - tp0) / (2 * K))
            pipelined = {"value": world * mp_per_step_rank / (p_ms / 1e3), "unit": "Mpixels/s", "ms_per_step": p_ms, "batches_in_flight": 2,
                         "note": "wall clock over %d decodes alternating between two resident batches on two streams" % (2 * K)}
            b2.close()
        except Exception as e:
            pipelined = {"value": None, "note": "failed: %r" % (e,)}
    # ---- bit-exactness of what was just timed: a sample for most workloads, EVERY image for verify_all workloads ----
    def reference_pixels(i):
        """tight reference image of unique image i: the compiled reference when it travelled, else the C restatement"""
        from oracle import refdrv
        if refdrv.available("sse"):
            ref = refdrv.Ref("sse")
            if pixel_type > J.EIGHT_BIT_GRAYSCALE:
                rc, err, img, _ = ref.decode_dither(jpegs[i], pixel_type, opt)
            else:
                rc, err, img, _ = ref.decode_cb(jpegs[i], pixel_type, opt, want_log=False)
            return (img if rc == 1 else None), "reference (oracle/_ref SSE2 build)"
        from tests import common as T
        rc, img = T.oracle_decode(jpegs[i], pixel_type, opt, 0, wl["w"], wl["h"])
        return (img if rc == 1 else None), "C restatement (oracle/jpegdec_oracle.c)"

    parity, parity_all = None, None
    try:
        if rank == 0:
            nchk = min(4, unique)
            okc, src = 0, ""
            for i in range(nchk):
                want, src = reference_pixels(i)
                got = b.read_output(i)
                okc += int(want is not None and got.shape[0] == oh0 and np.array_equal(got[:, :row_bytes], want[:oh0, :row_bytes]))
            parity = "%d/%d sampled images of the timed batch bit-exact vs %s" % (okc, nchk, src)
        if wl.get("verify_all"):
            # digests on the device (JPEGB200_digestDevice) of every image of this rank's batch vs digests of the reference's pixels
            want_d = []
            for i in range(unique):
                img, src = reference_pixels(i)
                want_d.append(J.digest_host(img[:oh0, :row_bytes]) if img is not None else None)
            devp = [b.device_output(i)[0] for i in range(n_img)]
            got_d = ctx.digest_device(devp, [oh0 * row_bytes] * n_img)
            good = sum(1 for i in range(n_img) if got_d[i] == want_d[i % unique])
            tot = torch.tensor([good, n_img], dtype=torch.int64, device="cuda")
            if world > 1:
                dist.all_reduce(tot)
            parity_all = {"verified": int(tot[0].item()), "images": int(tot[1].item()), "against": src,
                          "how": "64-bit digest of each image's device-resident pixels (JPEGB200_digestDevice) == digest of the reference's pixels for that seed"}
    except Exception as e:  # parity is asserted in tests/; here it is informational
        parity = "not checked: %r" % (e,)
    table_hits = ctx.shared_table_hits()
    b.close()

    # ---- one call per step, device outputs (verify_all workloads): JPEGB200_decodeBatch cuts the rank's slice into jobs ----
    dev_one_call = None
    if wl.get("verify_all"):
        per = oh0 * row_bytes
        stride = (per + 255) & ~255
        dev = ctx.device_alloc(stride * n_img)
        douts = [dev + i * stride for i in range(n_img)]

        def dev_call():
            rc, s2, c2 = J.decode_batch(ctx, ptrs, sizes, pixel_type, opt, douts, None, J.JPEGB200_OUT_DEVICE)
            if rc != 1:
                raise SystemExit("decodeBatch(OUT_DEVICE) failed: rc=%d %s" % (rc, s2[:8]))
            return c2
        for _ in range(max(1, min(W, 2))):
            dev_call()
        barrier()
        t0 = time.time()
        for _ in range(K):
            c2 = dev_call()
        barrier()
        t1 = time.time()
        oc_ms = max_over_ranks(1e3 * (t1 - t0) / K)
        tms, njobs = ctx.last_call_timings()
        got_d = ctx.digest_device(douts, [per] * n_img)
        good = sum(1 for i in range(n_img) if got_d[i] == want_d[i % unique])
        tot = torch.tensor([good, n_img], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(tot)
        dev_one_call = {"value": world * mp_per_step_rank / (oc_ms / 1e3), "unit": "Mpixels/s", "ms_per_step": oc_ms, "jobs_per_call": njobs,
                    "h2d_bytes_per_step": int(c2["h2d_bytes"]), "verified": int(tot[0].item()), "images": int(tot[1].item()),
                    "note": "ONE JPEGB200_decodeBatch(JPEGB200_OUT_DEVICE) call per rank and step: compressed files in pinned host memory "
                            "(H2D inside the timed region), pixels written to the caller's device buffer; wall clock, max over ranks"}
        ctx.device_free(dev)

    # ---- end to end through the public C ABI with host buffers (`e2e`) ----
    e2e = None
    if not args.no_e2e:
        out_bytes = oh0 * row_bytes
        stride = (out_bytes + 255) & ~255
        n_e2e = n_img
        try:   # the pinned output of every rank must fit the host (uhd10k: 20.7 GB per rank)
            avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0]
            while n_e2e > 64 and stride * n_e2e * world > 0.5 * avail:
                n_e2e //= 2
        except Exception:
            pass
        out_ptr = L.JPEGB200_hostAlloc(stride * n_e2e + 256)
        if out_ptr:
            outs = [out_ptr + i * stride for i in range(n_e2e)]

            def one_call():
                rc, s2, c2 = J.decode_batch(ctx, ptrs[:n_e2e], sizes[:n_e2e], pixel_type, opt, outs)
                if rc != 1:
                    raise SystemExit("e2e decodeBatch failed: rc=%d %s" % (rc, s2[:8]))
                return s2, c2
            for _ in range(max(1, min(W, 2))):
                one_call()
            barrier()
            t0 = time.time()
            for _ in range(K):
                s2, c2 = one_call()
            barrier()
            t1 = time.time()
            e_ms = max_over_ranks(1e3 * (t1 - t0) / K)
            e2e = {"value": world * (mp_per_step_rank * n_e2e / n_img) / (e_ms / 1e3), "unit": "Mpixels/s",
                   "h2d_bytes_per_step": int(c2["h2d_bytes"]), "d2h_bytes_per_step": int(c2["d2h_bytes"]),
                   "ms_per_step": e_ms, "images_per_gpu": n_e2e, "d2h_gb_per_s_per_gpu": float(c2["d2h_bytes"]) / (e_ms / 1e3) / 1e9,
                   "note": "one JPEGB200_decodeBatch C-ABI call per step, host buffers both sides (pinned): host parse + H2D + kernels + D2H of all pixels + status, run inside the call as a pipeline of 64-image jobs on separate streams"}
            L.JPEGB200_hostFree(out_ptr)
        else:
            e2e = {"value": None, "unit": "Mpixels/s", "note": "pinned output allocation failed"}
    L.JPEGB200_hostFree(in_ptr)

    # ---- roofline of the dominant kernel (fused IDCT + colour) ----
    peak, peak_src = load_peaks()
    alg_bytes = int(n_img * wl["w"] * wl["h"] * (wl["bpp_out"] + wl["coef_bpp"]))
    achieved = alg_bytes / (idct_ms / 1e3) / 1e9
    out_gbs = n_img * wl["w"] * wl["h"] * wl["bpp_out"] / (idct_ms / 1e3) / 1e9
    traffic, traffic_src = load_traffic(args.workload)
    roofline = {"bound": "hbm", "kernel": wl.get("kernel", "jdk_idct_tb / jdk_idct_color (fused expand + dequant + IDCT + colour)"), "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": idct_ms,
                "write_only_gbs": out_gbs, "write_frac": out_gbs / peak,
                "kernel_share_of_step": idct_ms / (dev_ms / K) if dev_ms > 0 else None,
                "dominant": bool(idct_ms >= entropy_ms),
                "note": "achieved = SURVEY 8(d) algorithmic bytes (output + 2 B x samples per source pixel) / CUDA-event time of the launch; "
                        "write_frac = output bytes only (the north-star's 0.40 target); traffic = ncu dram read + write of the named capture"}
    # the whole step against the same roof: compressed bytes in + pixels out (SURVEY 8(d) whole-pipeline figure)
    step_bytes = float(cnt["compressed_bytes"]) + float(cnt["output_bytes"])
    step_roofline = {"algorithmic_bytes_per_step": step_bytes, "achieved": step_bytes / ((dev_ms / K) / 1e3) / 1e9, "unit": "GB/s",
                     "frac": step_bytes / ((dev_ms / K) / 1e3) / 1e9 / peak,
                     "entropy_stage_ms": entropy_ms, "entropy_share_of_step": entropy_ms / (dev_ms / K) if dev_ms > 0 else None}

    # ---- CPU baseline beside it (rank 0, N=1 only, bounded sample) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and pixel_type <= J.EIGHT_BIT_GRAYSCALE:
        try:
            from oracle import refdrv
            os.sched_setaffinity(0, full_affinity)      # the reference gets every CPU the process may use, not just the GPU's node
            if refdrv.available("sse"):
                n_sample = max(threads * 8, 256)
                v, secs = cpu_reference_run(wl, jpegs, pixel_type, n_sample, threads, passes=3)
                v1, secs1 = cpu_reference_run(wl, jpegs, pixel_type, 32, 1, passes=2)
                cpu = {"value": v, "unit": "Mpixels/s", "cores": threads, "kind": "reference",
                       "sample": "%d images (%d unique cycled), best of 3, framebuffer mode, oracle/_ref SSE2 build" % (n_sample, unique),
                       "single_thread_value": v1, "host": cpu_facts}
        except Exception as e:
            cpu = {"value": None, "unit": "Mpixels/s", "cores": threads, "kind": "reference", "sample": "failed: %r" % (e,)}

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    if rank == 0:
        line = {
            "metric": "Mpixels/sec baseline 4:2:0 decode (batch)", "value": value, "unit": "Mpixels/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16/int32 (u8 pixels)", "data": "synthetic (%d unique seeds per GPU cycled to %d images)" % (unique, n_img),
            "config": config, "clocks": clocks, "gpu_launches": int(launches),
            "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu,
            "stages_ms": {k: v / K for k, v in stage.items()}, "wall_ms_per_step": wall_ms_step,
            "entropy_symbol_stage_ms": entropy_ms, "quirk_events_per_step": int(cnt["events"]),
            "shared_table_hits": table_hits, "parity_spot_check": parity, "parity_all": parity_all, "one_call_device": dev_one_call,
            "step_roofline": step_roofline, "numa": numa, "two_batches_in_flight": pipelined,
            "entropy_pipeline": os.environ.get("JPEGDEC_B200_ENTROPY", "clean (jdk_unstuff_segs + word reader)")}
        try:   # SURVEY.md 8(d): the entropy stage is reported as compressed MB/s; scaled workloads also as output pixels
            comp_mb = float(cnt["compressed_bytes"]) / 1e6
            line["entropy_compressed_mb_per_s"] = world * comp_mb / (entropy_ms / 1e3) if entropy_ms > 0 else None
            sh = {2: 1, 4: 2, 8: 3}.get(int(wl.get("opt", 0)) & 14, 0)
            if sh:
                ow, oh = (wl["w"] + (1 << sh) - 1) >> sh, (wl["h"] + (1 << sh) - 1) >> sh
                line["output_mpixels_per_s"] = value * (ow * oh) / float(wl["w"] * wl["h"])
        except Exception:
            pass
        print(json.dumps(line, default=str))
    return 0


if __name__ == "__main__":
    sys.exit(main())
