#!/usr/bin/env python
"""PNG encode on the device (ops.encode_png) against cv2.imencode in a thread pool of os.cpu_count() workers on the
same host, and warp_files with each encoder.  Never a bench number.

    python profiles/png_probe.py [out_dir]      # out_dir (default: a new temporary directory) receives the
                                                # warp_files output

Device encode is timed with CUDA events around the two launches over batches that rotate so that the inputs do not
fit the 126 MB L2; "to host" adds the offsets and payload copies of image_io.encode_png_device (wall clock).  Rates
are images/s and raw (uncompressed) GB/s."""
import concurrent.futures as cf
import io
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from attwarp_b200 import image_io, ops  # noqa: E402

dev = torch.device("cuda", 0)
gen = torch.Generator(device=dev).manual_seed(0)
WORKERS = os.cpu_count() or 1
L2_BYTES = 126 << 20


def photo_like(h, w):
    """tests/test_image_io.py::_photo_like, built on the device."""
    y = torch.arange(h, device=dev, dtype=torch.float64)[:, None].expand(h, w)
    x = torch.arange(w, device=dev, dtype=torch.float64)[None, :].expand(h, w)
    base = torch.stack([127 + 100 * torch.sin(x / 17 + y / 23), 127 + 90 * torch.cos(x / 11 - y / 29),
                        255 * (x + y) / (h + w)], -1)
    base += torch.randn(base.shape, device=dev, dtype=torch.float64, generator=gen) * 6
    base[h // 3: h // 2, w // 4: w // 2] = torch.tensor([230.0, 40.0, 60.0], device=dev, dtype=torch.float64)
    return base.round().clamp(0, 255).to(torch.uint8)


def noise(h, w):
    return torch.randint(0, 256, (h, w, 3), device=dev, dtype=torch.uint8, generator=gen)


def shapes(name):
    if name == "256 x 336^2":
        return [(336, 336)] * 256
    if name == "64 x 1344^2":
        return [(1344, 1344)] * 64
    rng = np.random.default_rng(0)          # 1024 mixed: sides 224 .. 1344, the drivers' 500^2 among them
    return [(int(h), int(w)) for h, w in rng.integers(224, 1345, (1024, 2))]


def time_device(batches, reps):
    for b in batches:                       # warm-up: every batch once
        ops.encode_png(b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        ops.encode_png(batches[r % len(batches)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def time_to_host(batch, reps=3):
    image_io.encode_png_device(batch)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        files = image_io.encode_png_device(batch)
    return (time.perf_counter() - t0) / reps, sum(len(f) for f in files)


def time_cv2(host_imgs):
    import cv2
    cv2.imencode(".png", host_imgs[0])
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(max_workers=WORKERS) as ex:
        sizes = list(ex.map(lambda im: len(cv2.imencode(".png", im)[1]), host_imgs))
    return time.perf_counter() - t0, sum(sizes)


def encode_rows():
    print(f"{'batch':14s} {'content':8s} {'raw MB':>8s} | {'device s':>9s} {'img/s':>9s} {'GB/s':>6s} | "
          f"{'to host s':>9s} {'img/s':>9s} | {'cv2 pool s':>10s} {'img/s':>8s} | {'dev/cv2':>7s} {'size/cv2':>8s}")
    for name in ("256 x 336^2", "64 x 1344^2", "1024 mixed"):
        shp = shapes(name)
        for content, make in (("photo", photo_like), ("noise", noise)):
            batch = [make(h, w) for h, w in shp]
            raw = sum(t.numel() for t in batch)
            copies = max(1, -(-2 * L2_BYTES // raw))          # rotation > 2 x L2
            batches = [batch] + [[t.clone() for t in batch] for _ in range(copies - 1)]
            reps = max(6, copies * 2)
            dev_s = time_device(batches, reps)
            host_s, dev_bytes = time_to_host(batch)
            host_imgs = [t.cpu().numpy() for t in batch]
            cv2_s, cv2_bytes = time_cv2(host_imgs)
            n = len(batch)
            print(f"{name:14s} {content:8s} {raw / 1e6:8.1f} | {dev_s:9.5f} {n / dev_s:9.0f} {raw / dev_s / 1e9:6.1f} | "
                  f"{host_s:9.4f} {n / host_s:9.0f} | {cv2_s:10.3f} {n / cv2_s:8.0f} | {cv2_s / host_s:7.1f} "
                  f"{dev_bytes / cv2_bytes:8.4f}", flush=True)
            del batches, batch, host_imgs
            torch.cuda.empty_cache()


def warp_files_rows(out_dir):
    from PIL import Image
    rng = np.random.default_rng(1)
    n = 256
    files = []
    for k in range(n):
        img = photo_like(336, 336).cpu().numpy()
        buf = io.BytesIO()
        Image.fromarray(img).save(buf, format="JPEG", quality=90)
        files.append(buf.getvalue())
    tok = torch.from_numpy((rng.random((n, 24, 24)) ** 3).astype(np.float32))
    out_sizes = [(500, 500)] * n
    print(f"\nwarp_files: {n} JPEG files 336^2 -> warped PNG files 500^2 under {out_dir}")
    for label, on_dev in (("cv2.imwrite pool", False), ("device encoder", True)):
        d = os.path.join(out_dir, "dev" if on_dev else "cv2")
        os.makedirs(d, exist_ok=True)
        paths = [os.path.join(d, f"{k}.png") for k in range(n)]
        image_io.warp_files(files[:8], tok[:8], paths[:8], out_sizes[:8], workers=WORKERS, on_device_png=on_dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ok = image_io.warp_files(files, tok, paths, out_sizes, workers=WORKERS, on_device_png=on_dev)
        s = time.perf_counter() - t0
        assert all(ok)
        total = sum(os.path.getsize(p) for p in paths)
        print(f"  {label:18s} {s:7.3f} s  {n / s:8.0f} files/s  {total / n / 1e3:7.1f} kB per file", flush=True)


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix="png_probe_")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"GPU: {q[0] if q else torch.cuda.get_device_name(dev)}   host: {WORKERS} CPUs (cv2 pool workers)")
    import cv2
    print(f"cv2 {cv2.__version__}, torch {torch.__version__}\n")
    encode_rows()
    warp_files_rows(out_dir)


if __name__ == "__main__":
    main()
