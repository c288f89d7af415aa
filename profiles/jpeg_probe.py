#!/usr/bin/env python
"""Exact JPEG decode on the device (ops.decode_jpeg) against the host paths that give the same pixels, and nvJPEG.
Never a bench number.

    python profiles/jpeg_probe.py

Three lists, encoded here with Pillow at quality 90, 4:2:0: 256 x 336^2 photo-like, 64 x 1344^2 photo-like, 1024
photo-like of mixed sides 224 .. 2048 (like c4).  For each list:
  kernels     the seven launches of one attwarp_decode_jpeg call (CUDA events; compressed bytes already on the device)
  device call ops.decode_jpeg: host parse, one upload of the compressed bytes from pinned memory, kernels, status sync
  exact=True  image_io.decode_jpeg_batch(exact=True): Pillow on one host thread, then the uploads
  pool16      Pillow in a 16-thread pool, then the uploads
  nvJPEG      torchvision.io.decode_jpeg(device='cuda') (not Pillow's pixels), with the BGR HWC conversion
Wall-clock times end in a device synchronisation; each is the median of `reps` runs after a warm-up."""
import concurrent.futures as cf
import ctypes as C
import io
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from attwarp_b200 import _lib, image_io, ops  # noqa: E402

dev = torch.device("cuda", 0)


def photo_like(h, w, rng):
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    img = np.stack([127 + 100 * np.sin(x / 17 + y / 23), 127 + 90 * np.cos(x / 11 - y / 29), 255 * (x + y) / (h + w)],
                   -1)
    img += rng.normal(0, 6, img.shape)
    img[h // 3:h // 2, w // 4:w // 2] = (230, 40, 60)
    return np.clip(img.round(), 0, 255).astype(np.uint8)


def make_list(name):
    from PIL import Image
    rng = np.random.default_rng(0)
    if name == "256 x 336^2":
        shapes = [(336, 336)] * 256
    elif name == "64 x 1344^2":
        shapes = [(1344, 1344)] * 64
    else:
        shapes = [(int(h), int(w)) for h, w in rng.integers(224, 2049, (1024, 2))]
    cache = {}
    files = []
    for h, w in shapes:
        if (h, w) not in cache or len(cache) < 64:
            img = photo_like(h, w, rng)
            buf = io.BytesIO()
            Image.fromarray(img).save(buf, "JPEG", quality=90)
            cache[(h, w)] = buf.getvalue()
        files.append(cache[(h, w)])
    return files


def median_time(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def kernel_time(files, reps):
    """CUDA events around attwarp_decode_jpeg with the compressed bytes already on the device."""
    lib = _lib.load()
    n = len(files)
    blob = np.frombuffer(b"".join(files), dtype=np.uint8).copy()
    d = torch.from_numpy(blob).to(dev)
    offs = np.concatenate([[0], np.cumsum([len(b) for b in files])])
    infos = [ops.jpeg_probe(b) for b in files]
    outs = [torch.empty((h, w, 3), dtype=torch.uint8, device=dev) for h, w, _, _ in infos]
    table = np.zeros(n, dtype=ops._JPEG_DTYPE)
    table["host"] = blob.ctypes.data + offs[:-1]
    table["dev"] = d.data_ptr() + offs[:-1]
    table["nbytes"] = [len(b) for b in files]
    table["dst"] = [t.data_ptr() for t in outs]
    table["H"] = [i[0] for i in infos]
    table["W"] = [i[1] for i in infos]
    tp = table.ctypes.data_as(C.c_void_p)
    ws = torch.empty(lib.attwarp_jpeg_workspace_bytes(tp, n), dtype=torch.uint8, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    st = _lib.current_stream(dev)

    def call():
        _lib.check(lib.attwarp_decode_jpeg(tp, n, _lib.ptr(ws), ws.numel(), _lib.ptr(status), st))

    call()
    torch.cuda.synchronize()
    assert not status.cpu().numpy().any()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps):
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return float(np.median(ts)), sum(int(np.prod(t.shape)) for t in outs)


def pool16(files):
    from PIL import Image

    def one(b):
        return np.ascontiguousarray(np.array(Image.open(io.BytesIO(b)).convert("RGB"))[..., ::-1])

    with cf.ThreadPoolExecutor(max_workers=16) as ex:
        arrs = list(ex.map(one, files))
    return [torch.from_numpy(a).to(dev, non_blocking=True) for a in arrs]


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"GPU: {q[0] if q else torch.cuda.get_device_name(dev)}   host: {os.cpu_count()} CPUs", flush=True)
    print(f"{'list':14s} {'MB in':>7s} {'Mpx':>7s} | {'kernels s':>9s} | {'device s':>9s} {'img/s':>8s} | "
          f"{'exact=True s':>12s} | {'pool16 s':>9s} | {'nvJPEG s':>9s} | {'exact/dev':>9s}")
    for name in ("256 x 336^2", "64 x 1344^2", "1024 mixed"):
        files = make_list(name)
        n = len(files)
        mb = sum(len(b) for b in files) / 1e6
        reps = 5 if n > 500 else 10
        k_s, px = kernel_time(files, reps)
        dev_s = median_time(lambda: ops.decode_jpeg(files, dev), reps)
        ex_s = median_time(lambda: image_io.decode_jpeg_batch(files, dev, exact=True), 3)
        pool_s = median_time(lambda: pool16(files), 3)
        nv_s = median_time(lambda: image_io.decode_jpeg_batch(files, dev), reps)
        print(f"{name:14s} {mb:7.1f} {px / 3e6:7.1f} | {k_s:9.4f} | {dev_s:9.4f} {n / dev_s:8.0f} | {ex_s:12.3f} | "
              f"{pool_s:9.3f} | {nv_s:9.4f} | {ex_s / dev_s:9.1f}", flush=True)


if __name__ == "__main__":
    main()
