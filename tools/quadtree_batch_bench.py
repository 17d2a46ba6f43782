"""Per-image encode / decode time of the quadtree batch entries (fic_encode_quadtree_batch, fic_decode_quadtree_batch)
against a loop of single calls (fic_encode_quadtree[_rgb], fic_decode_quadtree[_rgb]), with every batch stream and decode
checked against the loop's.

    python tools/quadtree_batch_bench.py OUT_DIR [--sizes 1,8,64,256] [--reps 3]

Host buffers (planes, streams, outputs) are page-locked with fic_pin_host_buffer.  For each configuration and batch size n
it records, per image, the host time of the synchronised calls (the median of --reps repetitions after one warm-up) and
the device time the library's events report (fic_get_timings total_ms, summed over the loop's calls); the engine AUTO
ran at each level for a batch of n (what fic_encode_batch_u8 runs on the level's geometry); and the GPU's name and power
limit, read in the same run.  Writes OUT_DIR/quadtree_batch_bench.json and exits 1 if any batch output differs from
the loop's.
"""
import argparse
import ctypes as C
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

GOLD = os.path.join(ROOT, "tests", "golden")
MSE = 25.0

CONFIGS = [  # name, image set, b_max, b_min, wk (0: every level's whole pool)
    ("LenaGrey 256^2 (16, 8) whole pool", "lena_grey", 16, 8, 0),
    ("LenaGrey 256^2 (16, 8) wk=2", "lena_grey", 16, 8, 2),
    ("LenaGrey 256^2 (16, 4) whole pool", "lena_grey", 16, 4, 0),
    ("LenaGrey 256^2 (16, 4) wk=2", "lena_grey", 16, 4, 2),
    ("LenaColored 256^2 (16, 8) whole pool", "lena_rgb", 16, 8, 0),
    ("LenaColored 256^2 (16, 8) wk=2", "lena_rgb", 16, 8, 2),
    ("structured grey 1024^2 (16, 8) whole pool", "structured_1024", 16, 8, 0),
]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")[:2]
    return {"gpu": name, "power_limit": power}


def image_set(kind, n):
    """n distinct images: Lena shifted by 8 pixels per image (rolled, mirrored every other image), or synth.structured
    with one seed per image."""
    if kind == "structured_1024":
        return np.ascontiguousarray(np.stack([synth.structured(1024, 1024, 100 + i) for i in range(n)]))
    if kind == "lena_grey":
        base = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    else:
        base = np.fromfile(os.path.join(GOLD, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3).transpose(2, 0, 1)
    out = []
    for i in range(n):
        p = np.roll(base, 8 * (i // 2), axis=-1)
        out.append(p[..., ::-1] if i % 2 else p)
    return np.ascontiguousarray(np.stack(out))


class Bench:
    def __init__(self, h, planes, b_max, b_min, wk):
        self.h, self.L = h, h._L
        self.planes, self.b_max, self.b_min, self.wk = planes, b_max, b_min, wk
        self.rgb = planes.ndim == 4
        self.n, self.H, self.W = planes.shape[0], planes.shape[-2], planes.shape[-1]
        self.mode = fic.FIC_MODE_RGB_QT if self.rgb else fic.FIC_MODE_GREY_QT
        bound = self.L.fic_quadtree_rgb_stream_bound if self.rgb else self.L.fic_quadtree_stream_bound
        self.stride = bound(self.W, self.H, b_max, b_min)
        self.streams = np.zeros(self.n * self.stride, np.uint8)
        self.loop_streams = np.zeros(self.n * self.stride, np.uint8)
        self.sizes = np.zeros(self.n, np.uintp)
        self.loop_sizes = np.zeros(self.n, np.uintp)
        self.out = np.zeros(planes.shape, np.uint8)
        self.loop_out = np.zeros(planes.shape, np.uint8)
        self.avg, self.loop_avg = np.zeros(self.n, np.float32), np.zeros(self.n, np.float32)
        self.it, self.loop_it = np.zeros(self.n, np.int32), np.zeros(self.n, np.int32)
        self.pinned = [planes, self.streams, self.loop_streams, self.out, self.loop_out]
        for a in self.pinned:
            h.pin(a)

    def close(self):
        for a in self.pinned:
            self.h.unpin(a)

    def p(self, a, off=0):
        return C.c_void_p(a.ctypes.data + off)

    def _check(self, rc):
        if rc:
            raise fic.FicError(rc, self.L.fic_last_error(self.h._h).decode())

    def encode_batch(self):
        self._check(self.L.fic_encode_quadtree_batch(self.h._h, self.mode, self.p(self.planes), self.n, self.W, self.H,
                                                     self.b_max, self.b_min, self.wk, MSE, self.p(self.streams),
                                                     self.stride, self.p(self.sizes)))
        return self.h.timings().total_ms

    def encode_loop(self):
        fn = self.L.fic_encode_quadtree_rgb if self.rgb else self.L.fic_encode_quadtree
        img = self.planes[0].nbytes
        ms = 0.0
        for i in range(self.n):
            size = C.c_size_t(0)
            self._check(fn(self.h._h, self.p(self.planes, i * img), self.W, self.H, self.b_max, self.b_min, self.wk, MSE,
                           self.p(self.loop_streams, i * self.stride), self.stride, C.byref(size)))
            self.loop_sizes[i] = size.value
            ms += self.h.timings().total_ms
        return ms

    def decode_batch(self):
        self._check(self.L.fic_decode_quadtree_batch(self.h._h, self.mode, self.n, self.p(self.streams), self.stride,
                                                     self.p(self.sizes), 50, self.p(self.out), self.p(self.avg),
                                                     self.p(self.it)))
        return self.h.timings().total_ms

    def decode_loop(self):
        fn = self.L.fic_decode_quadtree_rgb if self.rgb else self.L.fic_decode_quadtree
        img = self.planes[0].nbytes
        ms = 0.0
        for i in range(self.n):
            avg, it = C.c_float(0), C.c_int(0)
            self._check(fn(self.h._h, self.p(self.loop_streams, i * self.stride), int(self.loop_sizes[i]), 50,
                           self.p(self.loop_out, i * img), C.byref(avg), C.byref(it)))
            self.loop_avg[i], self.loop_it[i] = avg.value, it.value
            ms += self.h.timings().total_ms
        return ms

    def same(self):
        streams = all(self.sizes[i] == self.loop_sizes[i] and
                      (self.streams[i * self.stride:i * self.stride + int(self.sizes[i])] ==
                       self.loop_streams[i * self.stride:i * self.stride + int(self.sizes[i])]).all() for i in range(self.n))
        decodes = ((self.out == self.loop_out).all() and (self.it == self.loop_it).all() and
                   self.avg.tobytes() == self.loop_avg.tobytes())
        return bool(streams), bool(decodes)


def timed(fn, reps):
    fn()  # warm-up
    host, dev = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        dev.append(fn())
        host.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(host)), float(np.median(dev))


def level_engines(h, planes, b_max, b_min, wk):
    names = {fic.FIC_ENGINE_DIRECT: "DIRECT", fic.FIC_ENGINE_UMMA: "UMMA", fic.FIC_ENGINE_FUSED: "FUSED"}
    out = {}
    B, W = b_max, planes.shape[-1]
    while B >= b_min:
        h.encode_batch_u8(planes, B, wk or 2 * (W // B) - 3)
        out[str(B)] = names.get(h.timings().engine, "?")
        B //= 2
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--sizes", default="1,8,64,256")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    sizes = [int(x) for x in args.sizes.split(",")]
    h = fic.Handle(0)
    result = {"device": gpu_info(), "max_mse": MSE, "max_iters": 50, "reps": args.reps, "rows": []}
    ok = True
    for name, kind, b_max, b_min, wk in CONFIGS:
        for n in sizes:
            planes = image_set(kind, n)
            b = Bench(h, planes, b_max, b_min, wk)
            try:
                enc_b = timed(b.encode_batch, args.reps)
                enc_l = timed(b.encode_loop, args.reps)
                dec_b = timed(b.decode_batch, args.reps)
                dec_l = timed(b.decode_loop, args.reps)
                same_streams, same_decodes = b.same()
                engines = level_engines(h, planes, b_max, b_min, wk)
                leaves = [int(b.sizes[i]) for i in range(n)]
            finally:
                b.close()
            ok = ok and same_streams and same_decodes
            row = {
                "config": name, "n": n, "W": planes.shape[-1], "H": planes.shape[-2], "b_max": b_max, "b_min": b_min,
                "wk": wk, "auto_engine_per_level": engines,
                "encode_ms_per_image": {"batch_host": enc_b[0] / n, "loop_host": enc_l[0] / n,
                                        "batch_device": enc_b[1] / n, "loop_device": enc_l[1] / n},
                "decode_ms_per_image": {"batch_host": dec_b[0] / n, "loop_host": dec_l[0] / n,
                                        "batch_device": dec_b[1] / n, "loop_device": dec_l[1] / n},
                "mean_stream_bytes": float(np.mean(leaves)), "mean_iterations": float(np.mean(b.it)),
                "streams_equal": same_streams, "decodes_equal": same_decodes,
            }
            result["rows"].append(row)
            e, d = row["encode_ms_per_image"], row["decode_ms_per_image"]
            print(f"{name:44s} n={n:4d}  encode {e['batch_host']:.4f} vs {e['loop_host']:.4f} ms/img  "
                  f"decode {d['batch_host']:.4f} vs {d['loop_host']:.4f} ms/img  {engines}  "
                  f"{'ok' if same_streams and same_decodes else 'DIFFERENT'}", flush=True)
    result["all_equal"] = ok
    with open(os.path.join(args.out_dir, "quadtree_batch_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    h.close()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
