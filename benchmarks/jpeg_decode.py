"""JPEG files to a padded, resized, mean-subtracted batch: host decode against device decode.

Workload: 64 images at VOC raw sizes (long side 500, portrait and landscape: the img_wh of tests/golden/voc_gt_200.npz
scaled to a long side of 500), resized to those img_wh, every other one mirrored.  Two file sets, written by
cv2.imwrite into a temporary directory:
  natural   synthetic natural pixels (as benchmarks/ragged_images.py), quality 90, 4:2:0 -- what VOC files look like;
  noise     a white-noise texture over the same structure, quality 95, 4:2:0 -- high entropy, long Huffman codes.
Paths, each the median over `--reps` repetitions of CUDA events around `--iters` back-to-back calls, host work included:
  a_serial_imread   today's preprocessed_batch_device: serial cv2.imread, pack_images upload, ragged resize;
  b_pool_imread     the same with cv2.imread on a thread pool of os.cpu_count() workers;
  c_device_decode   preprocessed_batch_device on the path-backed images: file read, header inspection, one upload of
                    the compressed files, device decode, ragged resize (and the status check that guards the fallback);
  decode_call       frcnn_jpeg_decode alone, files already in pinned and device memory (host header parse included);
  decode_kernels    the sum of the jpeg_* kernels' device times per call, from torch.profiler in a separate pass.
H2D bytes per batch: raw pixels for a / b, compressed files for c.  Prints one JSON line (and writes it to --out).

    python benchmarks/jpeg_decode.py [--batch 64] [--iters 20] [--reps 7] [--out results/jpeg_decode.json]
"""
import argparse
import concurrent.futures as cf
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _natural(h, w, seed, noise=False):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = 127 + 80 * np.sin(xx / 17.0 + seed) * np.cos(yy / 23.0) + 30 * np.sin((xx + yy) / 5.0)
    sigma = 60 if noise else 12
    return np.clip(base[:, :, None] + rng.normal(0, sigma, (h, w, 3)) + np.array([10, -20, 5]), 0, 255).astype(np.uint8)


def _gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:       # the numbers stand without it, but say so
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import cv2
    import torch
    from faster_rcnn_b200 import _build, ops, shapes
    from faster_rcnn_b200.runtime import get_context, ptr
    if not torch.cuda.is_available():
        raise SystemExit("jpeg_decode.py measures on the GPU; no CUDA device found")
    _build.build()
    ctx = get_context()
    g = np.load(os.path.join(ROOT, "tests", "golden", "voc_gt_200.npz"))
    rng = np.random.default_rng(0)
    wh = g["img_wh"][rng.integers(0, len(g["img_wh"]), args.batch)].astype(np.int64)
    dst = [(int(h), int(w)) for w, h in wh]
    raw = [(int(round(h * 500 / max(h, w))), int(round(w * 500 / max(h, w)))) for h, w in dst]

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.iters):
                fn()
            t1.record()
            t1.synchronize()
            ms.append(t0.elapsed_time(t1) / args.iters)
        return round(float(np.median(ms)), 4)

    result = {"gpu": _gpu_info(), "batch": args.batch, "iters": args.iters, "reps": args.reps, "cpus": os.cpu_count()}
    pool = cf.ThreadPoolExecutor(os.cpu_count())
    with tempfile.TemporaryDirectory() as tmp:
        for name, noise, quality in (("natural_q90_420", False, 90), ("noise_q95_420", True, 95)):
            paths = []
            for b, (h, w) in enumerate(raw):
                p = os.path.join(tmp, "%s_%03d.jpg" % (name, b))
                cv2.imwrite(p, _natural(h, w, b, noise), [cv2.IMWRITE_JPEG_QUALITY, quality,
                                                           cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                                           cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420])
                paths.append(p)
            images = []
            for b, p in enumerate(paths):
                img = shapes.Image("i%d" % b, dst[b][1], dst[b][0], image_path=p)
                images.append(img.horizontal_flip() if b % 2 else img)

            def with_pixels(raws):
                return [shapes.Image(i.name, i.width, i.height, (), i.flipped, r, i.image_path) for i, r in zip(images, raws)]

            def path_a():
                return shapes.preprocessed_batch_device(with_pixels([cv2.imread(p) for p in paths]))

            def path_b():
                return shapes.preprocessed_batch_device(with_pixels(list(pool.map(cv2.imread, paths))))

            def path_c():
                return shapes.preprocessed_batch_device(images)

            want = path_a()[0]
            assert torch.equal(path_c()[0], want) and torch.equal(path_b()[0], want), "paths disagree"
            files = [open(p, "rb").read() for p in paths]
            arrays = [np.frombuffer(f, np.uint8) for f in files]
            nb = np.array([a.size for a in arrays], np.int64)
            foff = np.concatenate([[0], np.cumsum(nb)[:-1]]).astype(np.int64)
            pinned = torch.from_numpy(np.concatenate(arrays)).pin_memory()
            files_dev = pinned.to(ctx.device)
            hw = [ops.jpeg_supported(a) for a in arrays]
            n_out = np.array([h * w * 3 for h, w in hw], np.int64)
            ooff = torch.from_numpy(np.concatenate([[0], np.cumsum(n_out)[:-1]]).astype(np.int64)).to(ctx.device)
            out = torch.empty(int(n_out.sum()), dtype=torch.uint8, device=ctx.device)
            status = torch.empty(len(files), dtype=torch.int32, device=ctx.device)

            def decode_call():
                ctx.call("frcnn_jpeg_decode", ptr(pinned), ptr(files_dev), foff.ctypes.data_as(ctypes.c_void_p),
                         nb.ctypes.data_as(ctypes.c_void_p), len(files), ptr(out), ptr(ooff), out.numel(),
                         ptr(status))

            r = {"a_serial_imread_ms": timed(path_a), "b_pool_imread_ms": timed(path_b), "c_device_decode_ms": timed(path_c),
                 "decode_call_ms": timed(decode_call),
                 "h2d_bytes_raw_pixels": int(sum(h * w * 3 for h, w in raw)), "h2d_bytes_files": int(nb.sum())}
            assert (status.cpu().numpy() == 0).all()
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.iters):
                    decode_call()
                torch.cuda.synchronize()
            per = {}
            for e in prof.key_averages():
                if "jpeg_" in e.key:
                    k = e.key.split("jpeg_", 1)[1].split("_kernel")[0]
                    per[k] = round(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1000.0 / args.iters, 4)
            r["decode_kernels_ms"] = round(sum(per.values()), 4)
            r["kernel_ms"] = per
            result[name] = r
    pool.shutdown()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
