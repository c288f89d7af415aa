#!/usr/bin/env python
"""The attention overlay on the device (ops.attention_overlay), alone and followed by the device PNG encoder
(ops.encode_png), against save_warped_image's host expression (cv2 + NumPy) in a thread pool of os.cpu_count()
workers on the same host.  Never a bench number.

    python profiles/overlay_probe.py

Device times: CUDA events around the call (descriptor upload + two launches) over batches that rotate so that the
inputs do not fit the 126 MB L2; the per-kernel split comes from a separate torch.profiler pass.  Algorithmic
bytes per pixel: image (3) + attention (map: its item size; token maps: the tokens, once) + output (3); the
min/max launch's second read of a map is listed on its own.  The copy peak is a device-to-device copy of 1 GiB
measured in the same run."""
import concurrent.futures as cf
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from attwarp_b200 import ops  # noqa: E402

dev = torch.device("cuda", 0)
gen = torch.Generator(device=dev).manual_seed(0)
WORKERS = os.cpu_count() or 1
L2_BYTES = 126 << 20


def shapes(name):
    if name == "256 x 336^2":
        return [(336, 336)] * 256
    if name == "64 x 1344^2":
        return [(1344, 1344)] * 64
    rng = np.random.default_rng(0)          # c4-like: 1024 sides 224 .. 1344
    return [(int(h), int(w)) for h, w in rng.integers(224, 1345, (1024, 2))]


def make_batch(shp, kind, grid):
    imgs = [torch.randint(0, 256, (h, w, 3), device=dev, dtype=torch.uint8, generator=gen) for h, w in shp]
    if kind == "tokens":
        tok = torch.rand((len(shp), grid, grid), device=dev, generator=gen) ** 3
        return imgs, dict(tok=tok), len(shp) * grid * grid * 4, 0
    att = [torch.randint(0, 256, (h, w), device=dev, dtype=torch.uint8, generator=gen) for h, w in shp]
    nbytes = sum(a.numel() for a in att)
    return imgs, dict(att=att), nbytes, nbytes


def copy_peak():
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * a.numel() * 10 / (e0.elapsed_time(e1) / 1e3)


def time_events(fn, batches, reps):
    for b in batches:
        fn(b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        fn(batches[r % len(batches)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def kernel_split(fn, batch):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fn(batch)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "overlay_" in e.key:
            name = "minmax" if "minmax" in e.key else "blend"
            out[name] = out.get(name, 0.0) + e.device_time_total / 5      # us per call
    return out


def host_overlay(image, att, alpha=0.5):
    """save_warped_image's overlay lines (the map already at the image's size)."""
    import cv2
    in_h, in_w = image.shape[:2]
    att_r = cv2.resize(att.copy(), (in_w, in_h), interpolation=cv2.INTER_LINEAR)
    lo, hi = np.min(att_r), np.max(att_r)
    att_n = (att_r - lo) / (hi - lo) if hi > lo + 1e-9 else np.zeros_like(att_r)
    heat = cv2.applyColorMap((att_n * 255).astype(np.uint8), cv2.COLORMAP_JET)
    return cv2.addWeighted(heat, alpha, image, 1 - alpha, 0)


def time_host(imgs, atts, encode):
    import cv2

    def one(k):
        ov = host_overlay(imgs[k], atts[k])
        return len(cv2.imencode(".png", ov)[1]) if encode else ov.size

    one(0)
    t0 = time.perf_counter()
    with cf.ThreadPoolExecutor(max_workers=WORKERS) as ex:
        list(ex.map(one, range(len(imgs))))
    return (time.perf_counter() - t0) / len(imgs)


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"GPU: {q[0] if q else torch.cuda.get_device_name(dev)}   host: {WORKERS} CPUs (host pool workers)")
    peak = copy_peak()
    print(f"device-to-device copy peak (1 GiB, read + write): {peak / 1e9:.0f} GB/s\n")
    print(f"{'batch':14s} {'attention':12s} {'alg MB':>7s} {'+mm MB':>7s} | {'call us':>8s} {'GB/s':>6s} {'peak':>5s} | "
          f"{'minmax us':>9s} {'blend us':>8s} {'blend GB/s':>10s} | {'+png us':>8s} | "
          f"{'host ms/img':>11s} {'+imencode':>9s} | {'dev/host':>8s}")
    for name in ("256 x 336^2", "64 x 1344^2", "1024 mixed"):
        shp = shapes(name)
        for kind, grid in (("tokens", 24 if name != "64 x 1344^2" else 48), ("u8 map", 0)):
            imgs, kw, att_bytes, mm_bytes = make_batch(shp, kind, grid)
            px = sum(h * w for h, w in shp)
            alg = px * 3 + att_bytes + px * 3
            copies = max(1, -(-2 * L2_BYTES // (alg + mm_bytes)))
            batches = [(imgs, kw)]
            for _ in range(copies - 1):
                batches.append(([t.clone() for t in imgs], {k: ([a.clone() for a in v] if isinstance(v, list) else v.clone())
                                                           for k, v in kw.items()}))
            reps = max(10, 2 * copies)
            ov = lambda b: ops.attention_overlay(b[0], **b[1])                      # noqa: E731
            ov_png = lambda b: ops.encode_png(ops.attention_overlay(b[0], **b[1]))  # noqa: E731
            call_s = time_events(ov, batches, reps)
            split = kernel_split(ov, batches[0])
            png_s = time_events(ov_png, batches, max(4, copies))
            n_host = {"256 x 336^2": 64, "64 x 1344^2": 16}.get(name, 64)
            h_imgs = [t.cpu().numpy() for t in imgs[:n_host]]
            if kind == "tokens":
                from oracle.numpy_path import upsample_tokens_nearest
                tok = kw["tok"][:n_host].cpu().numpy()
                h_atts = [upsample_tokens_nearest(tok[k], *h_imgs[k].shape[:2]) for k in range(n_host)]
            else:
                h_atts = [a.cpu().numpy() for a in kw["att"][:n_host]]
            host_s = time_host(h_imgs, h_atts, False)
            host_png_s = time_host(h_imgs, h_atts, True)
            blend_us = split.get("blend", float("nan"))
            print(f"{name:14s} {kind + (f' {grid}^2' if grid else ''):12s} {alg / 1e6:7.1f} {mm_bytes / 1e6:7.1f} | "
                  f"{call_s * 1e6:8.1f} {alg / call_s / 1e9:6.0f} {(alg + mm_bytes) / call_s / peak:5.2f} | "
                  f"{split.get('minmax', float('nan')):9.1f} {blend_us:8.1f} {alg / (blend_us * 1e-6) / 1e9:10.0f} | "
                  f"{png_s * 1e6:8.0f} | {host_s * 1e3:11.2f} {host_png_s * 1e3:9.2f} | "
                  f"{host_s * len(shp) / call_s:8.0f}", flush=True)
            del batches, imgs, kw
            torch.cuda.empty_cache()
    print("\npeak = (algorithmic bytes + the min/max re-read) / call time / copy peak; dev/host = the host pool's time "
          "for the whole batch over the device call's")


if __name__ == "__main__":
    main()
