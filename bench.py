#!/usr/bin/env python
"""bench.py -- encode throughput of the fractal encoder hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--size S] [--block B] [--pattern structured|noise] [--dump-outputs DIR]

One "step" = one full encode (pool build + range x domain search + code solve) of one
synthetic greyscale image with the whole domain pool as the search window
(widthKernel = domain blocks per width), BASELINE.json configs[2]/[3]:
    N = 1 : 4096 x 4096, B = 8 (the reference's default block size), 1 B200
    N > 1 : 8192 x 8192, B = 8, range-block rows sharded over N B200s, NCCL image broadcast
`value` is range x candidate evaluations per second of the whole job (inputs resident in
HBM); `mpixel_per_s` is the same time expressed as image pixels.  `e2e` is the same metric
through the C ABI with pinned HOST buffers (H2D of the image and D2H of the codes inside
the timed region).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
# DRAM bytes (read + write) of one k_umma_search launch from `ncu --set full` (profiles/), by (kind, size, B)
TRAFFIC = {("i8", 4096, 8): 1428918000, ("f16", 4096, 8): 651115008, ("f16_pair", 4096, 8): 659304704}
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=0, help="image edge; default 4096 (N=1) / 8192 (N>1)")
    ap.add_argument("--block", type=int, default=8)
    ap.add_argument("--pattern", default="structured", choices=["structured", "noise"])
    ap.add_argument("--engine", default="auto", choices=["auto", "direct", "umma"])
    ap.add_argument("--iso", action="store_true",
                    help="isometry extension: 8 isometries per candidate domain (8x the evaluations; not a reference mode)")
    ap.add_argument("--rgb", action="store_true",
                    help="RGB encode (FC:171-226: one shared domain and contrast for the three channels); tensor cores for B = 4, 8")
    ap.add_argument("--mma", default="auto", choices=["auto", "i8", "f16"],
                    help="tensor-core instruction kind of the tcgen05 search (auto: f16 for B=4,8; i8 for B=16)")
    ap.add_argument("--pair", default="auto", choices=["auto", "on", "off"],
                    help="CTA pairs (tcgen05 cta_group::2) of the tcgen05 search; auto = pairs at B = 8")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lena", action="store_true", help="skip the bundled-image object (BASELINE configs[0], [1], [4])")
    ap.add_argument("--parity-ranges", type=int, default=128,
                    help="range blocks of the timed result compared with the CPU oracle after the timed loop (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the codes of the last timed step to DIR/*.npy (--impl ours), so that two builds can be "
                         "compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


DUMP_LIMIT = 64 << 20   # bytes of all arrays --dump-outputs writes


def dump_outputs(out_dir, info, q, seed=2026):
    """Writes what a caller of the timed encode receives: info.npy (imageInfo floats, float32) and codes.npy (the
    writeData ints, as float64, which holds every int32 exactly).  Above DUMP_LIMIT a fixed, seeded sample of range
    blocks is written instead, with their indices in rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"info": np.asarray(info, np.float32), "codes": np.asarray(q, np.float64)}
    NR = info.shape[0]
    row_bytes = sum(a.itemsize * a.shape[1] for a in arrays.values())
    if NR * row_bytes > DUMP_LIMIT:
        n = (DUMP_LIMIT - 4096) // (row_bytes + 8)   # 8: the float64 row index; 4096: room for the .npy headers
        rows = np.sort(np.random.default_rng(seed).choice(NR, n, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def workload(args):
    size = args.size or (4096 if args.gpus == 1 else 8192)
    B = args.block
    wk = 2 * size // B - 3
    NR = (size // B) ** 2
    ND = wk * wk
    return size, B, wk, NR, ND


def make_image(args, size):
    import fractal_image_compression_b200 as fic

    gen = fic.synth.structured if args.pattern == "structured" else fic.synth.noise
    if args.rgb:   # three planes (R, G, B), seeds 1..3
        return np.stack([gen(size, size, s) for s in (1, 2, 3)], 0)
    return gen(size, size, 1)


def to_argb(plane):
    import fractal_image_compression_b200 as fic

    if plane.ndim == 2:
        return fic.synth.grey_to_argb(plane)
    v = plane.astype(np.uint32)
    return (np.uint32(0xFF000000) | (v[0] << np.uint32(16)) | (v[1] << np.uint32(8)) | v[2]).view(np.int32)


# ----------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference (the Java encoder cannot run: no JVM here)
# ----------------------------------------------------------------------------------------

def cpu_sample(plane, B, wk, nthreads, target_s, iso=False, rgb=False):
    """Times the oracle's range loop on the first R ranges of the workload.  The codebook
    build is timed separately (a call with zero ranges) and subtracted, so the figure is
    the search rate the reference would sustain over the full image."""
    from oracle import oracle as O
    import fractal_image_compression_b200 as fic

    argb = to_argb(plane)
    kw = {"rgb": True} if rgb else {"iso": iso}
    t0 = time.perf_counter()
    O.encode(argb, B, wk, range_begin=0, range_end=0, nthreads=1, **kw)
    t_pool = time.perf_counter() - t0
    R = nthreads
    t0 = time.perf_counter()
    O.encode(argb, B, wk, range_begin=0, range_end=R, nthreads=nthreads, **kw)
    t_probe = max(time.perf_counter() - t0 - t_pool, 1e-3)
    R = max(nthreads, int(R * target_s / t_probe) // nthreads * nthreads)
    R = min(R, (argb.shape[0] // B) * (argb.shape[1] // B))   # small images: the whole image is the sample
    t0 = time.perf_counter()
    O.encode(argb, B, wk, range_begin=0, range_end=R, nthreads=nthreads, **kw)
    t = max(time.perf_counter() - t0 - t_pool, 1e-6)
    return R, t, t_pool


def parity_spot(plane, B, wk, info, q, K, iso=False, rgb=False, seed=2026):
    """Untimed check of the result the timed loop produced: K random range blocks plus the first and the last one,
    recomputed by the CPU oracle (oracle/, the C restatement of FC:613-644 / FC:655-687 / FC:697-808) on all host
    threads and compared bit for bit -- the unquantised floats of imageInfo[RGB] and the ints writeData emits."""
    from oracle import oracle as O

    argb = to_argb(plane)
    NR = info.shape[0]
    rng = np.random.default_rng(seed)
    ranges = np.unique(np.concatenate([[0, NR - 1], rng.integers(0, NR, K)])).astype(np.int64)
    t0 = time.perf_counter()
    ref = O.encode_list(argb, B, wk, ranges, rgb=rgb, iso=iso, nthreads=os.cpu_count() or 1)
    t_cpu = time.perf_counter() - t0
    got = np.ascontiguousarray(info[ranges])
    # floats must agree bit for bit; a NaN contrast (0/0 on a flat winner, FC:634) must be NaN on both sides
    same_f = (got.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(got) & np.isnan(ref))
    scale = {3: (1, 100, 1), 5: (1, 1000000, 100000, 100000, 1), 4: (1, 100, 1, 1)}[info.shape[1]]
    with np.errstate(invalid="ignore", over="ignore"):
        refq = np.stack([java_f2i(ref[:, c] * np.float32(scale[c])) for c in range(info.shape[1])], 1)
    same_q = q[ranges] == refq
    bad = int((~(same_f.all(1) & same_q.all(1))).sum())
    return {"ranges": int(len(ranges)), "mismatches": bad, "checker": "oracle", "oracle_seconds": round(t_cpu, 2),
            "compared": "imageInfo floats (bitwise) and writeData ints"}


def java_f2i(x):
    """Java (int)float: truncate toward zero, saturate, NaN -> 0 (FC:242-244, FC:250-254)."""
    x = np.asarray(x, np.float32)
    out = np.zeros(x.shape, np.int32)
    ok = ~np.isnan(x)
    xc = np.clip(np.trunc(np.where(ok, x, 0).astype(np.float64)), -2147483648.0, 2147483647.0)
    out[ok] = xc[ok].astype(np.int64).astype(np.int32)
    return out


def lena_object(handle, fic):
    """BASELINE configs[0], [1], [4]: the bundled Lena images (decoded pixels: tests/golden/) through the
    reference-shaped host entries -- ARGB ints in, codes out, decode back to ARGB -- beside the single-threaded oracle.
    Not part of the timed metric.  GPU times are the library's own event pair around each call (copies included),
    best of 20 calls after 3 warm-ups; `*_equals_oracle` compare the byte stream writeData would emit."""
    from oracle import oracle as O

    gold = os.path.join(ROOT, "tests", "golden")
    grey = np.fromfile(os.path.join(gold, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    l64 = np.fromfile(os.path.join(gold, "lena64.u8"), np.uint8).reshape(64, 64)
    col = np.fromfile(os.path.join(gold, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3)
    with open(os.path.join(gold, "unknown_run.bin"), "rb") as f:
        unknown_run = f.read()
    cases = [("LenaGrey 256x256 B=8 wk=2 (reference defaults, configs[0])", to_argb(grey), 8, 2, False),
             ("LenaGrey 256x256 B=8 full pool (wk=61)", to_argb(grey), 8, 61, False),
             ("Lena64 64x64 B=8 wk=2 (configs[1])", to_argb(l64), 8, 2, False),
             ("Lena64 64x64 B=8 full pool (wk=13)", to_argb(l64), 8, 13, False),
             ("LenaColored 256x256 B=8 wk=2 RGB (configs[4], the reference's unknown.run)", to_argb(np.moveaxis(col, 2, 0)), 8, 2, True)]
    out = []
    engines = {fic.FIC_ENGINE_DIRECT: "direct", fic.FIC_ENGINE_UMMA: "tcgen05", fic.FIC_ENGINE_FUSED: "fused"}
    for name, argb, B, wk, rgb in cases:
        H, W = argb.shape
        S = 5 if rgb else 3
        NR = (W // B) * (H // B)
        info = np.zeros((NR, S), np.float32)
        q = np.zeros((NR, S), np.int32)
        dec = np.empty((H, W), np.int32)
        for a in (argb, info, q, dec):
            handle.pin(a)
        try:
            enc_ms, dec_ms = [], []
            for i in range(23):
                handle.encode(argb, B, wk, rgb=rgb, info=info, q=q)
                t = handle.timings()
                if i >= 3:
                    enc_ms.append(t.total_ms)
            engine = engines.get(t.engine, str(t.engine))
            for i in range(23):
                _, avg, iters = handle.decode(q, W, H, B, wk, rgb, out=dec)
                if i >= 3:
                    dec_ms.append(handle.timings().total_ms)
            t0 = time.perf_counter()
            handle.encode(argb, B, wk, rgb=rgb, info=info, q=q)
            enc_wall = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            handle.decode(q, W, H, B, wk, rgb, out=dec)
            dec_wall = (time.perf_counter() - t0) * 1e3
        finally:
            for a in (argb, info, q, dec):
                handle.unpin(a)
        t0 = time.perf_counter()
        oinfo = O.encode(argb, B, wk, rgb=rgb, nthreads=1)
        cpu_enc = (time.perf_counter() - t0) * 1e3
        ostream = O.write_data(oinfo, W, H, B, wk, rgb=rgb)
        t0 = time.perf_counter()
        oimg, oavg, oit = O.decode(ostream)
        cpu_dec = (time.perf_counter() - t0) * 1e3
        stream = fic.stream_write(q, W, H, B, wk, rgb)
        du, src = dec.view(np.uint32), argb.view(np.uint32)
        chans = (16, 8, 0) if rgb else (16,)
        mse = float(np.mean([(((du >> sh) & 0xFF).astype(np.float64) - ((src >> sh) & 0xFF)) ** 2 for sh in chans]))
        row = {"case": name, "engine": engine, "gpu_encode_ms": min(enc_ms), "gpu_decode_ms": min(dec_ms),
               "gpu_encode_ms_host_clock": enc_wall, "gpu_decode_ms_host_clock": dec_wall,
               "cpu_encode_ms_1thread": cpu_enc, "cpu_decode_ms_1thread": cpu_dec,
               "stream_equals_oracle": stream == ostream,
               "decode_equals_oracle": bool((dec == oimg).all() and np.float32(avg) == oavg and iters == oit),
               "iterations": int(iters), "avg_error": float(avg), "psnr_db": 10 * np.log10(255.0 ** 2 / max(mse, 1e-12))}
        if "unknown.run" in name:
            row["stream_equals_reference_unknown_run"] = stream == unknown_run
        out.append(row)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    size, B, wk, NR, ND = workload(args)
    plane = make_image(args, size)
    threads = os.cpu_count() or 1
    n_iso = 8 if args.iso else 1
    per_step = max(1.0, min(10.0, 100.0 / max(1, args.steps + args.warmup)))
    rates, times = [], []
    R = 0
    for i in range(args.warmup + args.steps):
        R, t, t_pool = cpu_sample(plane, B, wk, threads, per_step, args.iso, args.rgb)
        if i >= args.warmup:
            rates.append(R * ND * n_iso / t)
            times.append(t)
    v = statistics.mean(rates)
    full_s = NR * ND * n_iso / v
    line = {
        "impl": "reference", "metric": "encode_evals_per_s", "value": v / 1e9, "unit": "Gevals/s",
        "mpixel_per_s": size * size / full_s / 1e6,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": statistics.mean(times) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"synthetic {args.pattern} {size}x{size} {'RGB' if args.rgb else 'grey'}, B={B}, widthKernel={wk} (full pool)",
                   "ranges": NR, "domains": ND},
        "cpu_baseline": {"value": v / 1e9, "unit": "Gevals/s", "cores": threads, "kind": "port",
                         "sample": f"first {R} of {NR} range blocks against the full pool per step "
                                   f"(C restatement of the reference; JVM unavailable; codebook build excluded)"},
        "e2e": {"value": v / 1e9, "unit": "Gevals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------

def run_ours(args):
    import torch
    import torch.distributed as dist

    import fractal_image_compression_b200 as fic
    from fractal_image_compression_b200.dist import ShardedEncoder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    size, B, wk, NR, ND = workload(args)
    plane = make_image(args, size)
    n_iso = 8 if args.iso else 1
    if args.iso and args.rgb:
        raise SystemExit("--iso and --rgb exclude each other (the isometry extension is grey only)")
    mode = fic.FIC_MODE_GREY_ISO if args.iso else (fic.FIC_MODE_RGB if args.rgb else fic.FIC_MODE_GREY)
    S = 4 if args.iso else (5 if args.rgb else 3)
    C = 3 if args.rgb else 1
    evals = float(NR) * float(ND) * n_iso

    handle = fic.Handle(local)
    handle.set_engine({"auto": fic.FIC_ENGINE_AUTO, "direct": fic.FIC_ENGINE_DIRECT, "umma": fic.FIC_ENGINE_UMMA}[args.engine])
    handle.set_umma_kind({"auto": fic.FIC_UMMA_KIND_AUTO, "i8": fic.FIC_UMMA_KIND_I8, "f16": fic.FIC_UMMA_KIND_F16}[args.mma])
    handle.set_umma_pair({"auto": fic.FIC_UMMA_PAIR_AUTO, "on": fic.FIC_UMMA_PAIR_ON, "off": fic.FIC_UMMA_PAIR_OFF}[args.pair])
    # what the library runs: RGB has a kind::f16 path only; grey B = 16 a kind::i8 path only
    mma = "f16" if args.rgb else ("i8" if (B == 16 or args.mma == "i8") else "f16")
    stream = torch.cuda.Stream(dev)   # library work, NCCL ordering and the timing events all use this stream
    torch.cuda.set_stream(stream)
    handle.set_stream(stream.cuda_stream)
    enc = ShardedEncoder(handle=handle) if world > 1 else None

    d_planes = torch.from_numpy(plane).to(dev).reshape(C, size, size).contiguous() if rank == 0 else None
    d_info = torch.empty((NR, S), dtype=torch.float32, device=dev)
    d_q = torch.empty((NR, S), dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # pinned host buffers for the e2e leg
    h_argb = torch.from_numpy(to_argb(plane)).pin_memory() if rank == 0 else None
    h_plane = torch.from_numpy(plane).pin_memory() if rank == 0 else None
    h_info = torch.empty((NR, S), dtype=torch.float32).pin_memory()
    h_q = torch.empty((NR, S), dtype=torch.int32).pin_memory()

    last_out = [None, None]

    def step_device():
        if world == 1:
            handle.encode_planes_dev(d_planes.data_ptr(), mode, size, size, B, wk, 0, NR, d_info.data_ptr(), d_q.data_ptr())
            return None
        out = enc.encode(d_planes, mode, size, size, B, wk, device=dev)
        if out is not None:
            last_out[0], last_out[1] = out
        return out

    def step_e2e():
        if world == 1:
            # the call a user of the library makes: host ARGB in, host codes out
            handle.set_stream(None)
            handle.encode(h_argb.numpy(), B, wk, rgb=mode, info=h_info.numpy(), q=h_q.numpy())
            handle.set_stream(stream.cuda_stream)
            return
        pl = h_plane.to(dev, non_blocking=True).reshape(C, size, size) if rank == 0 else None
        out = enc.encode(pl, mode, size, size, B, wk, device=dev)
        if rank == 0:
            h_info.copy_(out[0], non_blocking=True)
            h_q.copy_(out[1], non_blocking=True)
        torch.cuda.synchronize(dev)

    def step_e2e_u8():
        # the same call for a host that already holds 8-bit pixels (fic_encode_grey_u8 / fic_encode_rgb_planes)
        handle.set_stream(None)
        handle.encode_u8(h_plane.numpy() if args.rgb else h_plane.numpy().reshape(size, size), B, wk, info=h_info.numpy(), q=h_q.numpy())
        handle.set_stream(stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, device_events):
        total_ms = 0.0
        kernel_ms, launches, search_ms, pool_ms = [], 0, [], []
        for _ in range(steps):
            flush.fill_(1)  # evict L2 between timed iterations (not timed)
            barrier()
            if device_events:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                torch.cuda.synchronize(dev)
                total_ms += e0.elapsed_time(e1)
            else:
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize(dev)
                total_ms += (time.perf_counter() - t0) * 1e3
            t = handle.timings()
            kernel_ms.append(t.kernel_ms)
            search_ms.append(t.search_ms)
            pool_ms.append(t.pool_ms)
            launches += t.launches
            barrier()
        return total_ms, kernel_ms, search_ms, pool_ms, launches

    for _ in range(max(args.warmup, 3)):
        step_device()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local)
    sampler.start()
    total_ms, kernel_ms, search_ms, pool_ms, launches = timed(step_device, args.steps, True)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        res_info, res_q = (d_info, d_q) if world == 1 else last_out
        dump_outputs(args.dump_outputs, res_info.cpu().numpy(), res_q.cpu().numpy())
    t = handle.timings()
    engine = t.engine
    step_evals = t.search_evals  # this rank's evaluations per step
    pair_used = handle.umma_pair_used()

    for _ in range(2):
        step_e2e()
    e2e_ms, _, _, _, e2e_launches = timed(step_e2e, args.steps, False)

    def lib_stages():
        """The library's own device-side event stamps of the last host-buffer call (copies included)."""
        tt = handle.timings()
        return {"h2d": tt.h2d_ms, "pool": tt.pool_ms, "search": tt.search_ms, "solve": tt.solve_ms, "d2h": tt.d2h_ms, "total": tt.total_ms}

    e2e_stages = lib_stages() if world == 1 else None
    e2e_u8_ms = e2e_u8_stages = None
    if world == 1 and not args.iso:
        step_e2e_u8()
        e2e_u8_ms, _, _, _, _ = timed(step_e2e_u8, args.steps, False)
        e2e_u8_stages = lib_stages()

    if world > 1:
        agg = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms = agg.tolist()
        nl = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(nl)
        launches = int(nl.item())
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = total_ms / args.steps
    value = evals / (ms_per_step * 1e-3)
    pk, pk_kind = peaks()
    k_ms = statistics.mean(kernel_ms)
    # Roofline of the dominant kernel.  MEASURED_PEAKS.json carries the cuBLAS bf16 rate (burst figure: the
    # kernel is timed alone by its own events); kind::f16 runs at the bf16 rate, kind::i8 at twice that.
    # A bare tcgen05.mma loop of the same kind and MMA shape is measured live as a second denominator.
    f16_peak = float(pk["bf16_tflops"])
    peak = f16_peak if mma == "f16" else 2.0 * f16_peak
    try:
        handle.set_stream(None)
        kk = fic.FIC_UMMA_KIND_F16 if mma == "f16" else fic.FIC_UMMA_KIND_I8
        bare = handle.measure_mma_peak_pair(kk) if pair_used else handle.measure_mma_peak(kk, 128)
    except Exception as exc:  # diagnostics only
        bare = None
        sys.stderr.write(f"tensor peak measurement failed: {exc}\n")
    try:
        bare_i8 = bare if mma == "i8" else handle.measure_mma_peak(fic.FIC_UMMA_KIND_I8, 128)
    except Exception as exc:
        bare_i8 = None
        sys.stderr.write(f"int8 peak measurement failed: {exc}\n")
    ops = 2.0 * B * B * step_evals       # algorithmic ops of one launch (SURVEY 8d: 2*B^2 per evaluation)
    achieved = ops / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
    nominal = 2250.0 if mma == "f16" else 4500.0
    is_umma = engine == fic.FIC_ENGINE_UMMA
    # The tensor pipe's own ceiling at the clock the GPU actually held during the timed steps (nvidia-smi samples):
    # 8192 (kind::f16) / 16384 (kind::i8) dense operations per clock and SM.  Both measured peaks above are taken under
    # the board's power cap with random operands; the search's operands are small integers and toggle less, so the
    # kernel can exceed them -- the per-clock ceiling is the one it cannot.
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    sm_mhz = clocks.get("sm_mhz") if isinstance(clocks, dict) else None
    pipe_at_clock = (8192.0 if mma == "f16" else 16384.0) * n_sm * float(sm_mhz) * 1e6 / 1e12 if sm_mhz else None
    roofline = {
        "bound": "tensor", "kernel": (f"k_umma_search (tcgen05.mma{'.cta_group::2' if pair_used else ''}.kind::{mma})" if is_umma
                                      else ("k_search_direct_rgb" if args.rgb else "k_search_direct_grey")),
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s" if mma == "f16" else "TOP/s", "frac": achieved / peak,
        "peak_source": (f"bf16_tflops ({pk['bf16_tflops']}, burst) of {pk_kind}" if mma == "f16" else
                        f"2 x bf16_tflops ({pk['bf16_tflops']}, burst) of {pk_kind} (no int8 entry there)"),
        "frac_of_nominal": achieved / nominal, "nominal": nominal,
        "bare_mma_loop_measured": bare,
        "bare_mma_loop_shape": "cta_group::2 M=256 N=128" if pair_used else "cta_group::1 M=128 N=128",
        "frac_of_bare_mma_loop": (achieved / bare) if bare else None,
        "pipe_peak_at_sampled_clock": pipe_at_clock, "sampled_sm_mhz": sm_mhz,
        "frac_of_pipe_at_sampled_clock": (achieved / pipe_at_clock) if pipe_at_clock else None,
        # north_star quotes the int8 tensor pipe: the same algorithmic rate against its nominal dense peak and against
        # a bare kind::i8 tcgen05.mma loop measured in this run (whatever instruction kind the kernel itself issues)
        "frac_of_int8_nominal": achieved / 4500.0,
        "int8_bare_mma_loop_measured": bare_i8,
        "frac_of_int8_measured": (achieved / bare_i8) if bare_i8 else None,
        "kernel_ms": k_ms, "search_ms": statistics.mean(search_ms),
        "pool_ms": statistics.mean(pool_ms),
        # dram__bytes_read.sum + dram__bytes_write.sum of one k_umma_search launch from `ncu --set full`
        # (profiles/); only known for the profiled workload
        "traffic": TRAFFIC.get((mma + ("_pair" if pair_used else ""), size, B)) if (is_umma and world == 1 and not args.iso and not args.rgb) else None,
        "traffic_source": "constant from the ncu --set full capture of this kernel on this workload (profiles/), not measured in this run",
    }
    line = {
        "metric": "encode_evals_per_s", "value": value / 1e9, "unit": "Gevals/s",
        "mpixel_per_s": size * size / (ms_per_step * 1e-3) / 1e6,
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": f"synthetic {args.pattern} {size}x{size} {'RGB' if args.rgb else 'grey'}, B={B}, widthKernel={wk} (full pool)"
                               + (", 8 isometries per domain (extension)" if args.iso else ""),
                   "ranges": NR, "domains": ND, "isometries": n_iso, "engine": f"tcgen05 kind::{mma}" if engine == fic.FIC_ENGINE_UMMA else "direct",
                   "cta_pairs": bool(pair_used),
                   "parallelism": f"range-rows x{world}", "l2": "flushed between timed iterations (256 MiB write)",
                   # the library's once-per-handle check that kind::f16 accumulators are the exact integer covariances
                   "f16_exact_selftest": bool(handle.f16_exact()) if mma == "f16" else None},
        "clocks": clocks,
        "e2e": {"value": evals / (e2e_ms / args.steps * 1e-3) / 1e9, "unit": "Gevals/s",
                "mpixel_per_s": size * size / (e2e_ms / args.steps * 1e-3) / 1e6,
                "ms_per_step": e2e_ms / args.steps,
                "h2d_bytes_per_step": size * size * (4 if world == 1 else C), "d2h_bytes_per_step": NR * 8 * S,
                "entry": ("fic_encode_grey / fic_encode_rgb: the reference's int32 ARGB array in, imageInfo + writeData ints out"
                          if world == 1 else "8-bit planes in (rank 0), NCCL broadcast, fic_encode_planes_dev per rank, codes gathered to rank 0 and copied to the host")},
        "gpu_launches": launches,
        "roofline": roofline,
    }
    if e2e_stages is not None:
        line["e2e"]["device_stage_ms"] = e2e_stages   # ms_per_step above is the host clock around the call
    if e2e_u8_ms is not None:
        line["e2e_u8"] = {"value": evals / (e2e_u8_ms / args.steps * 1e-3) / 1e9, "unit": "Gevals/s", "ms_per_step": e2e_u8_ms / args.steps,
                          "h2d_bytes_per_step": size * size * C, "d2h_bytes_per_step": NR * 8 * S,
                          "entry": "fic_encode_grey_u8 / fic_encode_rgb_planes: 8-bit planes in, the same outputs",
                          "device_stage_ms": e2e_u8_stages}
    if world == 1:
        # verification leg (untimed part of the contract): the GPU decoder reconstructs the image from the
        # quantised codes just produced; PSNR against the source is what fractal coding reaches on this content
        h_q.copy_(d_q)
        q_host = h_q.numpy()
        h_dec = torch.empty((size, size), dtype=torch.int32).pin_memory()   # pinned like the encode leg's buffers
        handle.set_stream(None)
        handle.decode(q_host, size, size, B, wk, mode, out=h_dec.numpy())   # warm-up (allocations)
        t0 = time.perf_counter()
        dec, avg_err, iters = handle.decode(q_host, size, size, B, wk, mode, out=h_dec.numpy())
        t_dec = time.perf_counter() - t0
        dev_ms = handle.timings().total_ms
        du = dec.view(np.uint32)
        rec = (np.stack([(du >> 16) & 0xFF, (du >> 8) & 0xFF, du & 0xFF], 0) if args.rgb else ((du >> 16) & 0xFF)).astype(np.float64)
        mse = float(np.mean((rec - plane.astype(np.float64)) ** 2))
        line["decode"] = {"iterations": int(iters), "avg_error": float(avg_err), "psnr_db": 10 * np.log10(255.0 ** 2 / max(mse, 1e-12)),
                          "ms_total_host_clock": t_dec * 1e3, "device_ms": dev_ms, "entry": "fic_decode: codes from the host, int32 ARGB image to the host",
                          "mpixel_per_s_per_sweep": size * size * iters / max(dev_ms, 1e-9) / 1e3}
        if not args.iso:
            # the same decode with 8-bit planes out (a quarter of the download) and with device-resident codes and image
            h_pl = torch.empty((C, size, size), dtype=torch.uint8).pin_memory()
            pl_out = h_pl.numpy() if args.rgb else h_pl.numpy().reshape(size, size)
            handle.decode_u8(q_host, size, size, B, wk, mode, out=pl_out)
            out8, avg8, it8 = handle.decode_u8(q_host, size, size, B, wk, mode, out=pl_out)
            u8_ms = handle.timings().total_ms
            d_out = torch.empty((C, size, size), dtype=torch.uint8, device=dev)
            handle.decode_planes_dev(d_q.data_ptr(), size, size, B, wk, mode, d_out.data_ptr())
            avgd, itd = handle.decode_planes_dev(d_q.data_ptr(), size, size, B, wk, mode, d_out.data_ptr())
            dev_only_ms = handle.timings().total_ms
            same = bool((out8.reshape(C, size, size) == rec.astype(np.uint8).reshape(C, size, size)).all()
                        and (d_out.cpu().numpy() == out8.reshape(C, size, size)).all() and it8 == iters and itd == iters
                        and float(avg8) == float(avg_err) and float(avgd) == float(avg_err))
            sweep_bytes = 3.25 * size * size * C + 12.0 * NR   # SURVEY 8d: algorithmic bytes of one decoder sweep
            line["decode"].update({
                "device_ms_u8_planes_to_host": u8_ms, "device_ms_device_resident": dev_only_ms, "all_entries_agree": same,
                "sweep_us_device_resident": dev_only_ms * 1e3 / max(int(iters), 1),
                "sweep_hbm_roofline_frac": (sweep_bytes / (float(pk["hbm_gbs"]) * 1e9)) / (dev_only_ms * 1e-3 / max(int(iters), 1)),
                "sweep_roofline_note": "3.25*W*H*C + 12*NR bytes per sweep / measured copy bandwidth, against the whole device-resident call "
                                       "(code dequantisation, image fill and the skipped sweeps of the batch included) / iterations"})
    rc = 0
    if world == 1 and not args.no_lena:
        handle.set_stream(None)
        handle.set_engine(fic.FIC_ENGINE_AUTO)
        line["lena"] = lena_object(handle, fic)
        if not all(r["stream_equals_oracle"] and r["decode_equals_oracle"] and r.get("stream_equals_reference_unknown_run", True)
                   for r in line["lena"]):
            rc = 3
    if args.parity_ranges > 0:
        # the codes the timed loop left behind (the sharded, gathered result at N > 1) against the oracle
        if world == 1:
            res_info, res_q = d_info.cpu().numpy(), d_q.cpu().numpy()
        else:
            res_info, res_q = last_out[0].cpu().numpy(), last_out[1].cpu().numpy()
        line["parity_spot"] = parity_spot(plane, B, wk, res_info, res_q, args.parity_ranges, args.iso, args.rgb)
        if line["parity_spot"]["mismatches"]:
            rc = 3
    if world == 1 and not args.no_cpu_baseline:
        R, tcpu, t_pool = cpu_sample(plane, B, wk, 1, args.cpu_seconds, args.iso, args.rgb)
        v = R * ND * n_iso / tcpu
        line["cpu_baseline"] = {
            "value": v / 1e9, "unit": "Gevals/s", "cores": 1, "kind": "port",
            "host_cores": os.cpu_count(),
            "sample": f"first {R} of {NR} range blocks against the full pool, single thread like the reference "
                      f"(C restatement; JVM unavailable; codebook build {t_pool:.2f}s excluded)",
            "full_image_seconds_extrapolated": NR * ND * n_iso / v,
        }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if rc:
        sys.stderr.write("parity: a result differs from the oracle (parity_spot / lena)\n")
        sys.exit(rc)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
