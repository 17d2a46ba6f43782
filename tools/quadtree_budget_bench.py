"""The quadtree encode to a byte budget (fic_encode_quadtree_budget[_batch]) against the max_mse encode it replaces
(fic_encode_quadtree[_batch] at the m* the budget call chose), with every budget stream checked against that encode.

    python tools/quadtree_budget_bench.py OUT_DIR [--reps 5] [--quick]

Whole pool (wk = 0) throughout.  For each configuration it records the device time the library's events report
(fic_get_timings total_ms: the whole call, upload to last copy back), the median of --reps repetitions after one warm-up,
the budget call and the max_mse call alternating so that both see the same machine; the time of the budget form's own
kernels (k_qt_keys, k_qt_select) and of the split decision, from one torch.profiler run of their own; and a rate table on
LenaGrey and LenaColored 256^2: budget -> bytes, m* and decoded PSNR, beside the fixed B = 16 and B = 8 encodes.  The
GPU's name and power limit are read in the same run.  Writes OUT_DIR/quadtree_budget_bench.json; exits 1 if any budget
stream differs from the max_mse encode's at m*.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fractal_image_compression_b200 as fic  # noqa: E402
from fractal_image_compression_b200 import synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
NEW_KERNELS = ["k_qt_keys", "k_qt_select", "k_qt_decide"]


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


def lena(rgb):
    if rgb:
        return np.fromfile(os.path.join(GOLD, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3).transpose(2, 0, 1).copy()
    return np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)


def lena_set(rgb, n):
    """n distinct images: Lena rolled by 8 pixels per pair of images, mirrored every other image."""
    base, out = lena(rgb), []
    for i in range(n):
        p = np.roll(base, 8 * (i // 2), axis=-1)
        out.append(p[..., ::-1] if i % 2 else p)
    return np.ascontiguousarray(np.stack(out))


def extremes(shape, rgb, b_max, b_min):
    """(unsplit tree's size, fully split tree's size)."""
    H, W = shape[-2:]
    leaf, top = (20 if rgb else 12), (W // b_max) * (H // b_max)
    flags = (top + 3) & ~3
    return 32 + flags + leaf * top, 32 + flags + leaf * (W // b_min) * (H // b_min)


def compare(h, planes, rgb, b_max, b_min, budgets, reps):
    """Budget call vs the max_mse call at its m*, single (planes [H, W] / [3, H, W], one budget) or batch."""
    batch = planes.ndim == (4 if rgb else 3)
    if batch:
        budget = lambda: h.encode_quadtree_budget_batch(planes, b_max, b_min, 0, budgets)  # noqa: E731
    else:
        budget = lambda: h.encode_quadtree_budget(planes, b_max, b_min, 0, budgets)  # noqa: E731
    streams, mse = budget()
    if batch:  # the batch max_mse entry takes one max_mse: compare image by image, time the group at the median m*
        same = all(s == h.encode_quadtree(p, b_max, b_min, 0, float(m)) for s, p, m in zip(streams, planes, mse))
        m_ref = float(np.median(mse))
        ref = lambda: h.encode_quadtree_batch(planes, b_max, b_min, 0, m_ref)  # noqa: E731
        nbytes = float(np.mean([len(s) for s in streams]))
    else:
        same = streams == h.encode_quadtree(planes, b_max, b_min, 0, mse)
        ref = lambda: h.encode_quadtree(planes, b_max, b_min, 0, mse)  # noqa: E731
        nbytes = len(streams)
    tb, tr, lb, lr = [], [], 0, 0
    budget(), ref()  # warm-up
    for _ in range(reps):
        budget()
        t = h.timings()
        tb.append(t.total_ms)
        lb = t.launches
        ref()
        t = h.timings()
        tr.append(t.total_ms)
        lr = t.launches
    kb, nk = kernel_us(budget, NEW_KERNELS)
    return {"budget_ms": float(np.median(tb)), "max_mse_ms": float(np.median(tr)),
            "overhead_pct": 100.0 * (float(np.median(tb)) / float(np.median(tr)) - 1.0),
            "launches_budget": lb, "launches_max_mse": lr, "kernels_us": kb, "kernel_launches": nk,
            "mean_stream_bytes": nbytes, "max_mse": [float(m) for m in np.atleast_1d(mse)][:8], "streams_equal": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="skip the 4096^2 configurations")
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    import torch

    torch.cuda.init()
    h = fic.Handle(0)
    res = {"device": gpu_info(), "wk": 0, "reps": args.reps, "timing": [], "rate": []}
    ok = True
    configs = []
    for rgb in (False, True):
        for b_max, b_min in ((16, 8), (16, 4)):
            for n in (1, 64, 256):
                configs.append((f"{'LenaColored' if rgb else 'LenaGrey'} 256^2", rgb, b_max, b_min, n))
    if not args.quick:
        for b_max, b_min in ((16, 8), (16, 4)):
            configs.append(("structured grey 4096^2", False, b_max, b_min, 1))
    for name, rgb, b_max, b_min, n in configs:
        if name.startswith("structured"):
            planes = synth.structured(4096, 4096, 1)
        else:
            planes = lena(rgb) if n == 1 else lena_set(rgb, n)
        least, full = extremes(planes.shape, rgb, b_max, b_min)
        mid = (least + full) // 2
        budgets = mid if n == 1 else [least + (full - least) * (1 + i % 7) // 8 for i in range(n)]
        row = {"config": name, "n": n, "b_max": b_max, "b_min": b_min, "min_bytes": least, "full_bytes": full}
        row.update(compare(h, planes, rgb, b_max, b_min, budgets, args.reps))
        ok = ok and row["streams_equal"]
        res["timing"].append(row)
        print(json.dumps(row), flush=True)
    for rgb in (False, True):
        img = lena(rgb)
        for B in (16, 8):
            info, q = h.encode_u8(img, B, 2 * (256 // B) - 3)
            dec, _, _ = h.decode_u8(q, 256, 256, B, 2 * (256 // B) - 3, rgb)
            res["rate"].append({"image": "LenaColored" if rgb else "LenaGrey", "fixed_B": B, "bytes": 20 + (20 if rgb else 12) * len(q),
                                "psnr": psnr(dec, img)})
            print(json.dumps(res["rate"][-1]), flush=True)
        for b_max, b_min in ((16, 8), (16, 4)):
            least, full = extremes(img.shape, rgb, b_max, b_min)
            for frac in (0.0, 0.1, 0.2, 0.35, 0.5, 0.75, 1.0):
                budget = int(least + frac * (full - least))
                s, m = h.encode_quadtree_budget(img, b_max, b_min, 0, budget)
                same = s == h.encode_quadtree(img, b_max, b_min, 0, m)
                ok = ok and same
                dec, _, _ = h.decode_quadtree(s)
                res["rate"].append({"image": "LenaColored" if rgb else "LenaGrey", "b_max": b_max, "b_min": b_min, "budget": budget,
                                    "bytes": len(s), "max_mse": m, "psnr": psnr(dec, img), "stream_equal": bool(same)})
                print(json.dumps(res["rate"][-1]), flush=True)
    res["all_equal"] = bool(ok)
    with open(os.path.join(args.out_dir, "quadtree_budget_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    h.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
