"""Rate, quality and device time of the quadtree extension (FIC_MODE_GREY_QT, with --rgb FIC_MODE_RGB_QT) against the
fixed block sizes.

    python tools/quadtree_bench.py OUT_DIR [--quick] [--rgb]

Workloads: a structured synthetic 4096^2 image and LenaGrey 256^2 (--rgb: LenaColored 256^2 and a structured 2048^2 RGB
image, three synth.structured planes of different seeds; 2048^2 because the RGB B = 16 full pool has no tensor-core path
and every quadtree encode repeats it), quadtrees (16, 8) and (16, 4) with the whole pool and with widthKernel 2 over a
sweep of max_mse, and the fixed B = 16 / 8 / 4 encodes of the same images as baselines.
Per row: encode device ms (the call's total and its stages summed over levels), the quadtree kernels alone
(k_qt_collage_sse, k_qt_decide, k_qt_scatter: torch.profiler, one profiled call of its own), stream bytes and bits per
pixel, decode device ms, iterations, per-sweep kernel time, and PSNR against the source (RGB: over the 3*W*H samples).
Writes OUT_DIR/quadtree_bench.json (--rgb: quadtree_rgb_bench.json) with the GPU's name and power limit read in the same
run.  Exits 1 if a 256^2 stream does not decode through the CPU oracle to the GPU's pixels, iteration count and avgError.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import fractal_image_compression_b200 as fic  # noqa: E402
from oracle import quadtree as O  # noqa: E402
from oracle import quadtree_rgb as O_rgb  # noqa: E402

REPS = 5
MSES = [0.0, 4.0, 16.0, 36.0, 64.0, 100.0, 200.0, float("inf")]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")[:2]
    return {"gpu": name, "power_limit": power}


def psnr(a, b):
    mse = float(((a.astype(np.int64) - b.astype(np.int64)) ** 2).mean())
    return float("inf") if mse == 0 else 10.0 * np.log10(255.0 ** 2 / mse)


def kernel_us(fn, names):
    """Device time (us) of the kernels whose names contain one of `names`, in one profiled call of fn, and their count."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot, n = {}, {}
    for e in prof.events():
        dt = getattr(e, "device_time", None)
        if dt is None:
            dt = getattr(e, "cuda_time", 0.0)
        for k in names:
            if k in e.name and dt:
                tot[k] = tot.get(k, 0.0) + dt
                n[k] = n.get(k, 0) + 1
    return tot, n


def stages(t):
    return {"total_ms": t.total_ms, "pool_ms": t.pool_ms, "search_ms": t.search_ms, "kernel_ms": t.kernel_ms,
            "solve_ms": t.solve_ms, "engine": t.engine, "launches": t.launches}


def best(fn, h):
    ts = []
    for _ in range(REPS):
        out = fn()
        ts.append(h.timings())
    i = int(np.argmin([t.total_ms for t in ts]))
    return out, ts[i]


def main():
    out_dir = sys.argv[1]
    quick = "--quick" in sys.argv
    rgb = "--rgb" in sys.argv
    os.makedirs(out_dir, exist_ok=True)
    import torch

    torch.cuda.init()
    h = fic.Handle(0)
    if rgb:
        lena = np.fromfile(os.path.join(ROOT, "tests", "golden", "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3)
        images = {"lena_colored256": lena.transpose(2, 0, 1).copy()}
        if not quick:
            images["structured_rgb2048"] = np.stack([fic.synth.structured(2048, 2048, 1 + k) for k in range(3)])
        oracle_decode, code_bytes = O_rgb.decode_quadtree_rgb, 20
    else:
        lena = np.fromfile(os.path.join(ROOT, "tests", "golden", "lena_grey_256.u8"), np.uint8).reshape(256, 256)
        images = {"lena256": lena}
        if not quick:
            images["structured4096"] = fic.synth.structured(4096, 4096, 1)
        oracle_decode, code_bytes = O.decode_quadtree, 12
    res = {"device": gpu_info(), "reps": REPS, "fixed": [], "quadtree": []}
    failed = 0
    for name, plane in images.items():
        H, W = plane.shape[-2:]
        for wk in (0, 2):
            for B in (16, 8, 4):
                wkl = wk or 2 * (W // B) - 3
                (info, q), t = best(lambda: h.encode_u8(plane, B, wkl), h)
                (img, avg, it), td = best(lambda: h.decode_u8(q, W, H, B, wkl, rgb), h)
                sw, nsw = kernel_us(lambda: h.decode_u8(q, W, H, B, wkl, rgb), ["k_decode_sweep"])
                res["fixed"].append({"image": name, "B": B, "wk": wk, "encode": stages(t), "bytes": 20 + code_bytes * len(q),
                                     "bpp": (20 + code_bytes * len(q)) * 8 / (W * H), "decode_ms": td.total_ms, "iterations": it,
                                     "sweep_us": sum(sw.values()) / max(sum(nsw.values()), 1), "psnr": psnr(img, plane)})
                print(json.dumps(res["fixed"][-1]), flush=True)
            for b_max, b_min in ((16, 8), (16, 4)):
                for mse in MSES:
                    s, t = best(lambda: h.encode_quadtree(plane, b_max, b_min, wk, mse), h)
                    qk, _ = kernel_us(lambda: h.encode_quadtree(plane, b_max, b_min, wk, mse), ["k_qt_"])
                    (img, avg, it), td = best(lambda: h.decode_quadtree(s), h)
                    sw, nsw = kernel_us(lambda: h.decode_quadtree(s), ["k_decode_sweep_qt", "k_qt_dequant"])
                    row = {"image": name, "b_max": b_max, "b_min": b_min, "wk": wk, "max_mse": mse, "encode": stages(t),
                           "qt_kernels_ms": sum(qk.values()) / 1000.0, "bytes": len(s), "bpp": len(s) * 8 / (W * H),
                           "n_leaves": fic.quadtree_stream_info(s)[5], "decode_ms": td.total_ms, "iterations": it,
                           "avg_error": float(avg), "sweep_us": sw.get("k_decode_sweep_qt", 0.0) / max(nsw.get("k_decode_sweep_qt", 1), 1),
                           "psnr": psnr(img, plane)}
                    if W * H <= 256 * 256:
                        oimg, oavg, oit = oracle_decode(s)
                        row["oracle_roundtrip"] = bool((oimg == img).all() and oit == it and oavg.tobytes() == avg.tobytes())
                        failed += not row["oracle_roundtrip"]
                    res["quadtree"].append(row)
                    print(json.dumps(row), flush=True)
    h.close()
    res["oracle_roundtrip_failures"] = failed
    with open(os.path.join(out_dir, "quadtree_rgb_bench.json" if rgb else "quadtree_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
