#!/usr/bin/env python
"""PNG decode on the device (ops.decode_png) against the host paths that give the same pixels.  Never a bench
number.  Prints one JSON document; writes it to a file only with --out.

    python profiles/png_decode_probe.py [--out FILE] [--reps N]

Three lists of photo-like RGB images, each written three times (cv2.imencode at its default level, Pillow at
compress_level 6, and the cv2 files with their IDAT payloads joined into one chunk, as lodepng, stb_image_write or
the Rust png crate write them): 256 x 336^2, 64 x 1344^2, 1024 of mixed sides 224 .. 2048.  For each:
  kernels      one attwarp_decode_png call (CUDA events; the file bytes already on the device)
  device_call  ops.decode_png: host probe, pinned staging, one upload, the kernel, the status sync
  serial_cv2   today's exact_device loop for PNGs: cv2.imdecode file by file on one thread, each image uploaded
  pool16_cv2   cv2.imdecode in a 16-thread pool, then the uploads
Wall-clock times end in a device synchronisation; each is the median of `reps` runs after a warm-up (serial_cv2:
one run after a warm-up).  The card's
name, power limit and max SM clock are read in the same run."""
import argparse
import concurrent.futures as cf
import ctypes as C
import io
import json
import os
import struct
import subprocess
import sys
import time
import zlib

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from attwarp_b200 import _lib, ops  # noqa: E402

dev = torch.device("cuda", 0)
LISTS = ("256 x 336^2", "64 x 1344^2", "1024 mixed")


def photo_like(h, w, rng):
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.stack([127 + 100 * np.sin(x / 17 + y / 23), 127 + 90 * np.cos(x / 11 - y / 29), 255 * (x + y) / (h + w)],
                   -1)
    img += rng.normal(0, 6, img.shape).astype(np.float32)
    img[h // 3:h // 2, w // 4:w // 2] = (230, 40, 60)
    return np.clip(img.round(), 0, 255).astype(np.uint8)


def make_list(name, writer):
    from PIL import Image
    rng = np.random.default_rng(0)
    if name == LISTS[0]:
        shapes = [(336, 336)] * 256
    elif name == LISTS[1]:
        shapes = [(1344, 1344)] * 64
    else:
        shapes = [(int(h), int(w)) for h, w in rng.integers(224, 2049, (1024, 2))]
    seeds = rng.integers(0, 2**31, len(shapes))

    def one(k):
        img = photo_like(*shapes[k], np.random.default_rng(int(seeds[k])))
        if writer in ("cv2", "cv2_one_idat"):
            b = cv2.imencode(".png", img)[1].tobytes()
            return b if writer == "cv2" else one_idat(b)
        buf = io.BytesIO()
        Image.fromarray(img[..., ::-1]).save(buf, "PNG", compress_level=6)
        return buf.getvalue()

    with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 8) as ex:
        return list(ex.map(one, range(len(shapes))))


def one_idat(b):
    """The same file with its IDAT payloads joined into one chunk."""
    off, head, data, tail = 8, [], [], []
    while off < len(b):
        n, tag = struct.unpack(">I4s", b[off:off + 8])
        piece = b[off:off + 12 + n]
        if tag == b"IDAT":
            data.append(b[off + 8:off + 8 + n])
        elif data:
            tail.append(piece)
        else:
            head.append(piece)
        off += 12 + n
    data = b"".join(data)
    return (b[:8] + b"".join(head) + struct.pack(">I", len(data)) + b"IDAT" + data
            + struct.pack(">I", zlib.crc32(b"IDAT" + data)) + b"".join(tail))


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
    """CUDA events around attwarp_decode_png with the file bytes already on the device."""
    lib = _lib.load()
    n = len(files)
    blob = np.frombuffer(b"".join(files), dtype=np.uint8).copy()
    d = torch.from_numpy(blob).to(dev)
    offs = np.concatenate([[0], np.cumsum([len(b) for b in files])])
    infos = [ops.png_probe(b) for b in files]
    outs = [torch.empty((i[0], i[1], 3), dtype=torch.uint8, device=dev) for i in infos]
    table = np.zeros(n, dtype=ops._PNG_FILE_DTYPE)
    table["host"] = blob.ctypes.data + offs[:-1]
    table["dev"] = d.data_ptr() + offs[:-1]
    table["nbytes"] = [len(b) for b in files]
    table["dst"] = [t.data_ptr() for t in outs]
    table["H"] = [i[0] for i in infos]
    table["W"] = [i[1] for i in infos]
    tp = table.ctypes.data_as(C.c_void_p)
    ws = torch.empty(lib.attwarp_png_decode_workspace_bytes(tp, n), dtype=torch.uint8, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    st = _lib.current_stream(dev)

    def call():
        _lib.check(lib.attwarp_decode_png(tp, n, _lib.ptr(ws), ws.numel(), _lib.ptr(status), st))

    call()
    torch.cuda.synchronize()
    assert not status.cpu().numpy().any()
    for b, t in zip(files[:8], outs[:8]):
        assert np.array_equal(t.cpu().numpy(), cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps):
        e0.record()
        call()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return float(np.median(ts)), sum(int(np.prod(t.shape)) for t in outs)


def serial_cv2(files):
    return [torch.from_numpy(cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)).to(dev) for b in files]


def pool16(files):
    with cf.ThreadPoolExecutor(max_workers=16) as ex:
        arrs = list(ex.map(lambda b: cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR), files))
    return [torch.from_numpy(a).to(dev, non_blocking=True) for a in arrs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    fields = [f.strip() for f in q[0].split(",")] if q else [torch.cuda.get_device_name(dev), "unknown", "unknown"]
    doc = {"gpu": fields[0], "power_limit": fields[1], "max_sm_clock": fields[2], "host_cpus": os.cpu_count(),
           "rows": []}
    for name in LISTS:
        for writer in ("cv2", "pillow6", "cv2_one_idat"):
            files = make_list(name, writer)
            k_s, px = kernel_time(files, args.reps)
            row = {"list": name, "writer": writer, "files": len(files),
                   "mb_in": round(sum(len(b) for b in files) / 1e6, 1), "mpx": round(px / 3e6, 1),
                   "kernels_s": round(k_s, 5),
                   "device_call_s": round(median_time(lambda: ops.decode_png(files, dev), args.reps), 5),
                   "serial_cv2_s": round(median_time(lambda: serial_cv2(files), 1), 4),
                   "pool16_cv2_s": round(median_time(lambda: pool16(files), 3), 4)}
            row["pool16_over_device"] = round(row["pool16_cv2_s"] / row["device_call_s"], 2)
            doc["rows"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
