"""Per-image encode / decode time of the batch entries (fic_encode_batch[_u8], fic_decode_batch[_u8]) against a loop of
single calls, on images of the reference's own sizes, with every batch output checked against the loop's.

    python tools/batch_bench.py OUT_DIR [--sizes 1,8,64,256,1024] [--reps 3]

Host buffers are page-locked with fic_pin_host_buffer.  For each configuration and batch size n it records, per image:
device time (the library's events, fic_get_timings total_ms, summed over the loop's calls) and host time (a clock
around the synchronised call), for the ARGB and the 8-bit forms; the median of --reps repetitions after one warm-up.
Full-pool rows (widthKernel = domain blocks per side) also time the 8-bit batch with the engine forced to the tcgen05
group search and to the CUDA-core search, and record the engine AUTO ran: the data behind AUTO's batch rule.
Writes OUT_DIR/batch_bench.json and exits 1 if any batch output differs from the single-call loop.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fractal_image_compression_b200 as fic  # noqa: E402
from fractal_image_compression_b200 import synth  # noqa: E402

CONFIGS = [  # name, W, H, B, wk, rgb
    ("grey 256^2 B=8 wk=2 (reference default)", 256, 256, 8, 2, False),
    ("RGB 256^2 B=8 wk=2", 256, 256, 8, 2, True),
    ("grey 64^2 B=8 wk=2", 64, 64, 8, 2, False),
    ("grey 256^2 B=8 wk=16", 256, 256, 8, 16, False),
    # the full domain pool (the best-quality encode): AUTO runs groups of 4 or more images as tcgen05 group searches
    # instead of the CUDA-core search; the last row is a pool small enough for the fused kernel, which AUTO keeps
    ("grey 256^2 B=8 wk=61 (full pool)", 256, 256, 8, 61, False),
    ("grey 256^2 B=16 wk=29 (full pool)", 256, 256, 16, 29, False),
    ("grey 128^2 B=4 wk=61 (full pool)", 128, 128, 4, 61, False),
    ("RGB 256^2 B=8 wk=61 (full pool)", 256, 256, 8, 61, True),
    ("grey 512^2 B=8 wk=125 (full pool)", 512, 512, 8, 125, False),
    ("grey 64^2 B=8 wk=13 (full pool, fused)", 64, 64, 8, 13, False),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the query is informative only
        return {"error": str(e)}


def images(W, H, n, rgb, seed0):
    """n distinct images: synth.structured and synth.noise alternately, each with its own seed."""
    out = []
    for i in range(n):
        make = synth.structured if i % 2 == 0 else synth.noise
        s = seed0 + 3 * i
        out.append(np.stack([make(W, H, s), make(W, H, s + 1), make(W, H, s + 2)]) if rgb else make(W, H, s))
    planes = np.ascontiguousarray(np.stack(out))  # [n, H, W] or [n, 3, H, W]
    v = planes.astype(np.uint32)
    if rgb:
        argb = (np.uint32(0xFF000000) | (v[:, 0] << 16) | (v[:, 1] << 8) | v[:, 2]).view(np.int32)
    else:
        argb = (np.uint32(0xFF000000) | (v << 16) | (v << 8) | v).view(np.int32)
    return np.ascontiguousarray(argb), planes


def timed(h, fn, reps):
    """Median (device ms, host ms) of fn() over reps runs after one warm-up; fn returns the device ms of its calls."""
    fn()
    dev, host = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        d = fn()
        host.append((time.perf_counter() - t0) * 1e3)
        dev.append(d)
    return float(np.median(dev)), float(np.median(host))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def run_config(h, name, W, H, B, wk, rgb, sizes, reps, seed0):
    S = 5 if rgb else 3
    nr = (W // B) * (H // B)
    nmax = max(sizes)
    argb_all, planes_all = images(W, H, nmax, rgb, seed0)
    rows, mismatches = [], 0
    for n in sizes:
        argb, planes = argb_all[:n], planes_all[:n]
        info = np.zeros((n, nr, S), np.float32)
        q = np.zeros((n, nr, S), np.int32)
        info1 = np.zeros_like(info)
        q1 = np.zeros_like(q)
        img = np.zeros((n, H, W), np.int32)
        img1 = np.zeros_like(img)
        pl = np.zeros(planes.shape, np.uint8)
        pl1 = np.zeros_like(pl)
        avg, it = np.zeros(n, np.float32), np.zeros(n, np.int32)
        avg1, it1 = np.zeros_like(avg), np.zeros_like(it)
        pinned = [argb, planes, info, q, info1, q1, img, img1, pl, pl1]
        for a in pinned:
            h.pin(a)
        try:
            def enc_batch():
                h.encode_batch(argb, B, wk, rgb, info=info, q=q)
                return h.timings().total_ms

            def enc_loop():
                d = 0.0
                for i in range(n):
                    h.encode(argb[i], B, wk, rgb, info=info1[i], q=q1[i])
                    d += h.timings().total_ms
                return d

            def enc_batch_u8():
                h.encode_batch_u8(planes, B, wk, rgb, info=info, q=q)
                return h.timings().total_ms

            def enc_loop_u8():
                d = 0.0
                for i in range(n):
                    h.encode_u8(planes[i], B, wk, info=info1[i], q=q1[i])
                    d += h.timings().total_ms
                return d

            def dec_batch():
                _, a, t = h.decode_batch(q, W, H, B, wk, rgb, out=img)
                avg[:], it[:] = a, t
                return h.timings().total_ms

            def dec_loop():
                d = 0.0
                for i in range(n):
                    _, a, t = h.decode(q[i], W, H, B, wk, rgb, out=img1[i])
                    avg1[i], it1[i] = a, t
                    d += h.timings().total_ms
                return d

            def dec_batch_u8():
                _, a, t = h.decode_batch_u8(q, W, H, B, wk, rgb, out=pl)
                avg[:], it[:] = a, t
                return h.timings().total_ms

            def dec_loop_u8():
                d = 0.0
                for i in range(n):
                    _, a, t = h.decode_u8(q[i], W, H, B, wk, rgb, out=pl1[i])
                    avg1[i], it1[i] = a, t
                    d += h.timings().total_ms
                return d

            r = {"config": name, "W": W, "H": H, "B": B, "wk": wk, "rgb": rgb, "n": n}
            bad = {}
            for form, fb, fl in (("argb", enc_batch, enc_loop), ("u8", enc_batch_u8, enc_loop_u8)):
                r[f"encode_{form}_batch_dev_ms"], r[f"encode_{form}_batch_host_ms"] = timed(h, fb, reps)
                if form == "argb":
                    r["encode_batch_engine"] = h.timings().engine
                r[f"encode_{form}_loop_dev_ms"], r[f"encode_{form}_loop_host_ms"] = timed(h, fl, reps)
                nan_b, nan_l = np.isnan(info), np.isnan(info1)
                bad[f"encode_{form}"] = int(((bits(info) != bits(info1)) & ~(nan_b & nan_l)).any(axis=(1, 2)).sum()
                                            + (q != q1).any(axis=(1, 2)).sum())
            if wk == 2 * (W // B) - 3 and wk == 2 * (H // B) - 3:
                for eng, label in ((fic.FIC_ENGINE_UMMA, "umma"), (fic.FIC_ENGINE_DIRECT, "direct")):
                    h.set_engine(eng)
                    try:
                        r[f"encode_u8_batch_{label}_dev_ms"], r[f"encode_u8_batch_{label}_host_ms"] = timed(h, enc_batch_u8, reps)
                    finally:
                        h.set_engine(fic.FIC_ENGINE_AUTO)
                    nan_b, nan_l = np.isnan(info), np.isnan(info1)
                    bad[f"encode_u8_{label}"] = int(((bits(info) != bits(info1)) & ~(nan_b & nan_l)).any(axis=(1, 2)).sum()
                                                    + (q != q1).any(axis=(1, 2)).sum())
            for form, fb, fl, ob, ol in (("argb", dec_batch, dec_loop, img, img1), ("u8", dec_batch_u8, dec_loop_u8, pl, pl1)):
                r[f"decode_{form}_batch_dev_ms"], r[f"decode_{form}_batch_host_ms"] = timed(h, fb, reps)
                r[f"decode_{form}_loop_dev_ms"], r[f"decode_{form}_loop_host_ms"] = timed(h, fl, reps)
                bad[f"decode_{form}"] = int((ob != ol).reshape(n, -1).any(axis=1).sum() + (bits(avg) != bits(avg1)).sum()
                                            + (it != it1).sum())
            r["iterations_mean"] = float(it.mean())
            r["mismatched_images"] = bad
            mismatches += sum(bad.values())
            for k in list(r):
                if k.endswith("_ms"):
                    r[k.replace("_ms", "_us_per_image")] = r[k] * 1e3 / n
            rows.append(r)
            print(f"{name:40s} n={n:5d}  per image (us, device / host):"
                  f"  enc batch {r['encode_argb_batch_dev_us_per_image']:7.2f} / {r['encode_argb_batch_host_us_per_image']:7.2f}"
                  f"  loop {r['encode_argb_loop_dev_us_per_image']:7.2f} / {r['encode_argb_loop_host_us_per_image']:7.2f}"
                  f"  | dec batch {r['decode_argb_batch_dev_us_per_image']:7.2f} / {r['decode_argb_batch_host_us_per_image']:7.2f}"
                  f"  loop {r['decode_argb_loop_dev_us_per_image']:7.2f} / {r['decode_argb_loop_host_us_per_image']:7.2f}"
                  f"  | u8 enc {r['encode_u8_batch_dev_us_per_image']:7.2f} / {r['encode_u8_loop_dev_us_per_image']:7.2f}"
                  + (f" (umma {r['encode_u8_batch_umma_dev_us_per_image']:7.2f} direct {r['encode_u8_batch_direct_dev_us_per_image']:7.2f})"
                     if "encode_u8_batch_umma_dev_ms" in r else "") +
                  f"  dec {r['decode_u8_batch_dev_us_per_image']:7.2f} / {r['decode_u8_loop_dev_us_per_image']:7.2f}"
                  f"  mismatches {sum(bad.values())}", flush=True)
        finally:
            for a in pinned:
                h.unpin(a)
    return rows, mismatches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--sizes", default="1,8,64,256,1024")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    sizes = [int(x) for x in args.sizes.split(",")]
    os.makedirs(args.out_dir, exist_ok=True)
    result = {"gpu": gpu_info(), "sizes": sizes, "reps": args.reps, "rows": []}
    print(json.dumps(result["gpu"]), flush=True)
    h = fic.Handle(0)
    total = 0
    try:
        for k, (name, W, H, B, wk, rgb) in enumerate(CONFIGS):
            rows, bad = run_config(h, name, W, H, B, wk, rgb, sizes, args.reps, seed0=1000 * (k + 1))
            result["rows"] += rows
            total += bad
    finally:
        h.close()
    result["mismatches"] = total
    with open(os.path.join(args.out_dir, "batch_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(f"mismatches: {total}")
    return 1 if total else 0


if __name__ == "__main__":
    sys.exit(main())
