#!/usr/bin/env python
"""The drivers' mask flow on a mixed-size list: ops.warp_ragged_from_mota_tokens (one revise_mask launch, one fused
LANCZOS + marginals launch, finish, stage 5) against the per-image loop it replaces (ops.mota_mask per image, then
ops.warp_ragged_from_attention on the masks).  Never a bench number.

Lists: c4 (1024 square images, sides 224..2048, as profiles/c4_probe.py) and 256 images of independent sides 224..672.
Device times: CUDA events around whole calls, rotating over as many image sets as it takes for their images in and
out to exceed twice the 126 MB L2 (one set each at these sizes: 9.3 GB and 297 MB).  Host times: one call with the GPU
idle at its start.  Kernel times: torch.profiler in a pass of its own; the fused kernel is set beside the uniform one
at 64 x 1344^2.  Algorithmic bytes of the fused launch: uint8 token masks in + float32 maps out.  The copy peak and
the card's name and power limit are read in the same run.

    python profiles/ragged_mota_probe.py [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from attwarp_b200 import ops  # noqa: E402

L2_BYTES = 126 << 20
dev = torch.device("cuda", 0)


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


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def make_list(name, gen):
    rng = np.random.default_rng(1237)
    if name == "c4":
        s = rng.integers(224, 2049, size=1024)
        hw = [(int(v), int(v)) for v in s]
    else:
        hw = [(int(h), int(w)) for h, w in rng.integers(224, 673, size=(256, 2))]
    px = sum(h * w for h, w in hw)
    sets = max(1, -(-2 * L2_BYTES // (2 * 3 * px)))         # images in + out of all sets >= 2 x L2
    imgs = [[torch.randint(0, 256, (h, w, 3), device=dev, dtype=torch.uint8, generator=gen) for h, w in hw]
            for _ in range(sets)]
    tok = [(torch.rand(len(hw), 24, 24, device=dev, generator=gen) ** 3).contiguous() for _ in range(sets)]
    return hw, imgs, tok


def new_call(tok, imgs):
    return ops.warp_ragged_from_mota_tokens(tok, imgs)


def loop_call(tok, imgs):
    masks = [ops.mota_mask(tok[i:i + 1], (im.shape[0], im.shape[1]))[0] for i, im in enumerate(imgs)]
    return ops.warp_ragged_from_attention(masks, imgs)


def device_ms(fn, tok, imgs, reps):
    for k in range(len(imgs)):
        fn(tok[k], imgs[k])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        fn(tok[r % len(imgs)], imgs[r % len(imgs)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def host_ms(fn, tok, imgs):
    best = float("inf")
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(tok[0], imgs[0])
        best = min(best, time.perf_counter() - t0)
    torch.cuda.synchronize()
    return best * 1e3


def kernel_us(fn, key, reps=5):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = sum(e.device_time_total for e in prof.key_averages() if key(e.key))
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the whole result as JSON to this file")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    gen = torch.Generator(device=dev).manual_seed(0)
    res = {"card": card(), "copy_peak_GBps": copy_peak() / 1e9, "lists": {}}
    # the uniform fused kernel at 64 x 1344^2 (maps_from_mota_tokens), its kernel time alone
    tok64 = (torch.rand(64, 24, 24, device=dev, generator=gen) ** 3).contiguous()
    ops.maps_from_mota_tokens(tok64, (1344, 1344))
    u_us = kernel_us(lambda: ops.maps_from_mota_tokens(tok64, (1344, 1344)),
                     lambda k: "resize_lanczos_up_mma_kernel" in k)
    res["uniform_64x1344"] = {"kernel_us": u_us, "us_per_MP": u_us / (64 * 1344 * 1344 / 1e6)}
    for name in ("c4", "mixed256"):
        hw, imgs, tok = make_list(name, gen)
        n, px = len(hw), sum(h * w for h, w in hw)
        # first call of a list: the coefficient tables of every new size are built and uploaded once
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        new_call(tok[0], imgs[0])
        torch.cuda.synchronize()
        first_ms = (time.perf_counter() - t0) * 1e3
        r = {"n": n, "sets": len(imgs), "megapixels": px / 1e6, "first_call_ms": first_ms}
        r["new_device_ms"] = device_ms(new_call, tok, imgs, a.reps)
        r["loop_device_ms"] = device_ms(loop_call, tok, imgs, max(2, a.reps // 3))
        r["new_host_ms"] = host_ms(new_call, tok, imgs)
        r["loop_host_ms"] = host_ms(loop_call, tok, imgs)
        from attwarp_b200 import _lib
        new_call(tok[0], imgs[0])
        r["new_launches"] = int(_lib.load().attwarp_ragged_last_launches()) + 1      # + revise_mask
        k_us = kernel_us(lambda: new_call(tok[0], imgs[0]), lambda k: "resize_lanczos_up_mma_ragged_kernel" in k)
        alg = n * 24 * 24 + 4 * sum(h + w for h, w in hw)
        r["fused_kernel_us"] = k_us
        r["fused_us_per_MP"] = k_us / (px / 1e6)
        r["fused_vs_uniform_per_pixel"] = r["fused_us_per_MP"] / res["uniform_64x1344"]["us_per_MP"]
        r["fused_alg_bytes"] = alg
        r["fused_alg_GBps"] = alg / (k_us * 1e-6) / 1e9 if k_us > 0 else None
        res["lists"][name] = r
        print(name, json.dumps(r), flush=True)
        del imgs, tok
        torch.cuda.empty_cache()
    print(json.dumps({k: v for k, v in res.items() if k != "lists"}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
